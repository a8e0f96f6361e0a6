"""Every instance of the PGS solve and of the pre-solve kernels against the oracle or against each
other.  egg_launch_solve_pgs_stream picks one of 30 instances of egg_pgs_stream_kernel<LPW, MINB,
ISO, F32> (lanes per world 1 / 2 / 4 / 8 / 16, M^-1 layout 0 / 1 / 2, FP64 or FP32 records), the
opt-in run format one of 8 instances of egg_pgs_runs_kernel<LPW, ISO>, and the narrowphase and
record assembly have instances by threads per world.  Small batches select only a few of them, so
every case forces its instance with the development overrides (read per batch by egg_create) and
checks through Batch.kernel_config() that the instance it names is the one that ran.

FP32 records are held to the tolerances of test_pgs_fp32_records_opt_in, except that at converging
settings a sweep count may differ by one where the oracle shows an exact last sweep or a near-tie
at the stopping tolerance (tests.helpers.stepwise_fp32).

Each case prints one line: kernel, LPW, ISO, precision, worlds compared with the oracle, worst
relative errors and the sweeps of one step (min / max)."""
import numpy as np
import pytest

from tests.helpers import stepwise, stepwise_fp32

pytestmark = pytest.mark.gpu

OVERRIDES = ("EGG_PGS_LPW", "EGG_PGS_MIN_WARPS_PER_SM", "EGG_PGS_RUNS", "EGG_PGS_RUN_CAP", "EGG_PGS_TARGET_CTAS",
             "EGG_COLLIDE_NT", "EGG_RECORDS_NT", "EGG_PGS_ISO")
RUNS = 3 | 16        # QUIRKS_REFERENCE | EGG_OPT_PGS_RUNS


@pytest.fixture(autouse=True)
def _no_overrides(monkeypatch):
    for k in OVERRIDES:
        monkeypatch.delenv(k, raising=False)


# ---------------------------------------------------------------------------------------------
# Scenes
def _inertia(scene, iso, seed):
    """Reach an M^-1 layout through the bodies: 0 anisotropic inertia, 1 isotropic with m and I
    different per body, 2 the scene's uniform cubes."""
    rng = np.random.default_rng(seed)
    W, n = scene["W"], scene["n"]
    if iso == 0:
        scene["I"] = np.zeros((W, n, 3, 3))
        idx = np.arange(3)
        scene["I"][:, :, idx, idx] = rng.uniform(0.01, 0.05, size=(W, n, 3))
    elif iso == 1:
        scene["m"] = rng.uniform(0.5, 2.0, size=(W, n))
        scene["I"] = np.eye(3) * rng.uniform(0.05, 0.2, size=(W, n, 1, 1))
    return scene


def _cairn_mix(W, iso=2, seed=61, lifted=None):
    """Five rocks per world, three kinds of world side by side: a heap of colliding rocks (w % 3 == 0),
    rocks lifted out of reach with no constraint at all (w % 3 == 1), and rocks resting apart on the
    ground with small velocities, whose solves converge before k_max and stop at the exact residual
    (w % 3 == 2).  `lifted` replaces the world kinds' lifted set."""
    import eggshell_b200 as E
    rng = np.random.default_rng(seed + 1)
    sc = E.scenes.cairn(W, rocks=5, zb=(0.1, 0.6), seed=seed)
    kind = np.arange(W) % 3
    up = (kind == 1) if lifted is None else np.isin(np.arange(W), lifted)
    slow = (kind == 2) & ~up if lifted is None else np.zeros(W, dtype=bool)
    sc["p"][up, :, 2] += 50.0
    sc["p"][up, :, 0] += 3.0 * np.arange(5)
    ns = int(slow.sum())
    sc["p"][slow, :, 0] = -1.2 + 0.6 * np.arange(5) + rng.uniform(-0.03, 0.03, size=(ns, 5))
    sc["p"][slow, :, 1] = rng.uniform(-0.5, 0.5, size=(ns, 5))
    sc["p"][slow, :, 2] = rng.uniform(0.12, 0.16, size=(ns, 5))
    sc["v"][slow] *= 0.05
    sc["w"][slow] *= 0.05
    return _inertia(sc, iso, seed + 2)


def _scene(name, W, iso=2, seed=None):
    import eggshell_b200 as E
    if name == "cairn":
        return _cairn_mix(W, iso)
    sc = getattr(E.scenes, name)(W) if seed is None else getattr(E.scenes, name)(W, seed=seed)
    return _inertia(sc, iso, 71)


def _cairn40(W, seed=81):
    """40 rocks spread over a 3 m x 3 m box: a pile, not a block of interpenetrating rocks.  780
    pairs, so its narrowphase default is egg_collide_kernel<128>."""
    import eggshell_b200 as E
    return E.scenes.cairn(W, rocks=40, xb=(-1.5, 1.5), yb=(-1.5, 1.5), zb=(0.15, 1.2), seed=seed)


# ---------------------------------------------------------------------------------------------
# Instance checks
def _probe(scene, batch_kw):
    """The instance a batch of this scene and these settings runs (the overrides in the environment
    are read by egg_create, the M^-1 layout and the record format at the first step), and the sweeps
    of that first step."""
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, **batch_kw)
    b.step(scene["dt"])
    cfg, sw = b.kernel_config(), b.status()["sweeps"].copy()
    b.close()
    return cfg, sw


def _kernel(cfg):
    if cfg["rec_format"] == 2:
        return f"egg_pgs_runs_kernel<{cfg['lpw']},{cfg['iso']}> run cap {cfg['run_cap']}"
    minb = 8 if cfg["iso"] == 0 else 12
    return f"egg_pgs_stream_kernel<{cfg['lpw']},{minb},{cfg['iso']},{str(cfg['precision'] == 32).lower()}>"


def _report(what, cfg, nworlds, worst, sw):
    errs = " ".join(f"{k} {worst[k]:.1e}" for k in ("p", "R", "v", "w", "lam") if k in worst)
    for k in ("exact_sweep_plus_one", "near_tie"):
        if k in worst:
            errs += f" | {k.replace('_', ' ')}: {worst[k]} world-steps"
    print(f"{_kernel(cfg)} LPW {cfg['lpw']} ISO {cfg['iso']} FP{cfg['precision']} | {what}: {nworlds} worlds vs oracle | {errs} | "
          f"sweeps {int(sw.min())}/{int(sw.max())}")


def _oracle_case(monkeypatch, scene, steps, k_max, lpw, iso, prec, quirks=3, env=()):
    """Forces LPW (and `env`), checks the instance, then compares every world with the oracle step by
    step from shared state: FP64 at the tolerances of `stepwise`, FP32 records at 1e-4 with
    bit-exact narrowphase outputs and the sweep counts of `stepwise_fp32(sweep_slack=True)`."""
    import eggshell_b200 as E
    monkeypatch.setenv("EGG_PGS_LPW", str(lpw))
    for k, v in env:
        monkeypatch.setenv(k, v)
    kw = dict(solver=E.SOLVER_PGS, k_max=k_max, quirks=quirks)
    cfg, sw = _probe(scene, dict(kw, precision=prec))
    assert (cfg["lpw"], cfg["worlds_per_warp"], cfg["iso"], cfg["precision"]) == (lpw, 32 // lpw, iso, prec), cfg
    assert cfg["rec_format"] == (2 if quirks & 16 else 1), cfg
    idx = list(range(scene["W"]))
    if prec == 64:
        worst = stepwise(scene, steps, idx, kw, dict(solver=1, k_max=k_max))
    else:
        worst = stepwise_fp32(scene, steps, idx, kw, dict(solver=1, k_max=k_max), sweep_slack=True)
    _report(scene["name"], cfg, len(idx), worst, sw)
    return cfg, sw


# ---------------------------------------------------------------------------------------------
# (a) the 30 stream instances against the oracle
@pytest.mark.parametrize("prec", [64, 32])
@pytest.mark.parametrize("iso", [0, 1, 2])
@pytest.mark.parametrize("lpw", [1, 2, 4, 8, 16])
def test_stream_instance_vs_oracle(lpw, iso, prec, monkeypatch):
    """W = 2G + 3 worlds: two full warp groups and a ragged one.  The mixed cairn (colliding, lifted
    and converging worlds in one batch; at least one world stops before k_max) and legged20 (joints
    and contacts, k_max = 100), every world against the oracle."""
    W = 2 * (32 // lpw) + 3
    _, sw = _oracle_case(monkeypatch, _cairn_mix(W, iso), 4, 500, lpw, iso, prec)
    assert ((sw > 0) & (sw < 500)).any(), f"no world converged early: {sw.tolist()}"
    _oracle_case(monkeypatch, _scene("legged20", W, iso), 2, 100, lpw, iso, prec)


# ---------------------------------------------------------------------------------------------
# (b) the 8 run-format instances against the oracle
@pytest.mark.parametrize("iso", [1, 2])
@pytest.mark.parametrize("lpw", [1, 2, 4, 8])
def test_run_format_instance_vs_oracle(lpw, iso, monkeypatch):
    W = 2 * (32 // lpw) + 3
    _, sw = _oracle_case(monkeypatch, _cairn_mix(W, iso), 4, 500, lpw, iso, 64, quirks=RUNS)
    assert ((sw > 0) & (sw < 500)).any(), f"no world converged early: {sw.tolist()}"
    _oracle_case(monkeypatch, _scene("legged20", W, iso), 2, 100, lpw, iso, 64, quirks=RUNS)
    _oracle_case(monkeypatch, _scene("stack10", W, iso), 3, 500, lpw, iso, 64, quirks=RUNS)


def test_run_format_caps_vs_oracle(monkeypatch):
    """Runs spanning several stages: pile64 at K = 50, where the computed run cap (6) is below the 8
    lanes per world, and EGG_PGS_RUN_CAP = 1 on the stack and the cairn."""
    cfg, _ = _oracle_case(monkeypatch, _scene("pile64", 3), 2, 50, 8, 2, 64, quirks=RUNS)
    assert 0 < cfg["run_cap"] < cfg["lpw"], cfg
    for scene, steps in ((_scene("stack10", 11), 3), (_cairn_mix(11), 4)):
        cfg, _ = _oracle_case(monkeypatch, scene, steps, 500, 8, 2, 64, quirks=RUNS, env=(("EGG_PGS_RUN_CAP", "1"),))
        assert cfg["run_cap"] == 1, cfg


# ---------------------------------------------------------------------------------------------
# (c) bit identity across the stage cut
def _fixed_k_outputs(scene, k_max, maxc, monkeypatch, lpw, prec=64, quirks=3):
    import eggshell_b200 as E
    monkeypatch.setenv("EGG_PGS_LPW", str(lpw))
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, max_contacts=maxc, quirks=quirks, precision=prec)
    b.step(scene["dt"], n_steps=2)
    cfg = b.kernel_config()
    assert cfg["lpw"] == lpw and cfg["precision"] == prec and cfg["rec_format"] == (2 if quirks & 16 else 1), cfg
    st = b.status()
    assert int(np.bitwise_or.reduce(st["status"])) == 0
    con = b.contacts()
    out = dict(zip("pRvw", (x.copy() for x in b.bodies())), lam=con["lam"], row_state=con["row_state"],
               count=con["count"], sweeps=st["sweeps"].copy())
    b.close()
    return cfg, out


@pytest.mark.parametrize("name,W,k_max", [("stack10", 4000, 10), ("legged20", 4000, 10), ("pile64", 1000, 10), ("pile64", 1000, 500)])
def test_state_is_bit_identical_across_lanes_per_world(name, W, k_max, monkeypatch):
    """Blocks of one stage share no body, so they commute exactly (DESIGN.md, "Gauss-Seidel order and
    exactness"): the stage cut, i.e. the lanes per world, cannot change a bit of the state, the
    multipliers, the clamp states or the sweep counts.  Two steps at fixed K (no world converges, so
    the LPW-dependent order of the residual sum cannot move a sweep count), for FP64 records, FP32
    records and the run format across each one's lane counts."""
    scene = _scene(name, W)
    maxc = 1024 if name == "pile64" else 0
    for prec, quirks, lpws in ((64, 3, (1, 2, 4, 8, 16)), (32, 3, (1, 2, 4, 8, 16)), (64, RUNS, (1, 2, 4, 8))):
        ref = None
        for lpw in lpws:
            cfg, out = _fixed_k_outputs(scene, k_max, maxc, monkeypatch, lpw, prec, quirks)
            if ref is None:
                ref, ref_lpw = out, lpw
                assert int(out["sweeps"].max()) == k_max, "no world reached K: the case does not exercise the solve"
                continue
            for key, a in out.items():
                b = ref[key]
                assert np.array_equal(a.view(np.uint64) if a.dtype == np.float64 else a, b.view(np.uint64) if b.dtype == np.float64 else b), \
                    f"{name} K={k_max} {_kernel(cfg)}: {key} differs from LPW {ref_lpw} in {int(np.sum(np.any((a != b).reshape(W, -1), axis=1)))} worlds"
        print(f"{name} W={W} K={k_max} FP{prec} {'run format' if quirks & 16 else 'group stream'}: bit-identical across LPW {list(lpws)}")


# ---------------------------------------------------------------------------------------------
# (d) pre-solve instances: narrowphase and record assembly threads per world
def _presolve_outputs(scene, kw):
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, taps=True, **kw)
    b.step(scene["dt"], n_steps=2)
    cfg = b.kernel_config()
    assert int(np.bitwise_or.reduce(b.status()["status"])) == 0
    out = dict(b.contacts())
    out.update({"hit_" + k: v for k, v in b.pair_hits().items()})
    out.update(zip("pRvw", b.bodies()))
    b.close()
    return cfg, out


@pytest.mark.parametrize("name", ["pile64", "legged20", "cairn40"])
def test_presolve_instances_are_bit_identical(name, monkeypatch):
    """Forced narrowphase threads {32, 64, 128, 256} and record-assembly threads {32, 64, 128, 256}
    (run format: {32, 128, 256}) give the same contact lists, pair hits, contact geometry, multipliers
    and state bit for bit as the default instance."""
    import eggshell_b200 as E
    scene = _cairn40(8) if name == "cairn40" else _scene(name, 8)
    for quirks, var, values in ((3, "EGG_COLLIDE_NT", (32, 64, 128, 256)), (3, "EGG_RECORDS_NT", (32, 64, 128, 256)),
                                (RUNS, "EGG_RECORDS_NT", (32, 128, 256))):
        kw = dict(solver=E.SOLVER_PGS, k_max=20, quirks=quirks)
        monkeypatch.delenv(var, raising=False)
        dcfg, ref = _presolve_outputs(scene, kw)
        assert dcfg["rec_format"] == (2 if quirks & 16 else 1)
        slot = "collide_threads" if var == "EGG_COLLIDE_NT" else "records_threads"
        for nt in values:
            monkeypatch.setenv(var, str(nt))
            cfg, out = _presolve_outputs(scene, kw)
            assert cfg[slot] == nt, (var, nt, cfg)
            for key, a in out.items():
                assert np.array_equal(a, ref[key]), f"{name} {var}={nt}: {key} differs from the default ({dcfg[slot]} threads)"
        monkeypatch.delenv(var)
        what = "egg_collide_kernel" if var == "EGG_COLLIDE_NT" else ("egg_records_runs_kernel" if quirks & 16 else "egg_records_kernel")
        print(f"{name}: {what}<{'|'.join(map(str, values))}> bit-identical to the default <{dcfg[slot]}>, "
              f"{int(ref['count'].sum())} contacts, {int(ref['hit_n'].sum())} pair hits")


def test_cairn40_default_instances_vs_oracle():
    """The 40-rock cairn at its default instances (egg_collide_kernel<128>, egg_records_kernel<128>)
    stepwise against the oracle."""
    import eggshell_b200 as E
    scene = _cairn40(4)
    kw = dict(solver=E.SOLVER_PGS)
    cfg, sw = _probe(scene, kw)
    assert cfg["collide_threads"] == 128 and cfg["records_threads"] == 128, cfg
    worst = stepwise(scene, 3, list(range(4)), kw, dict(solver=1))
    _report("cairn40 egg_collide_kernel<128>", cfg, 4, worst, sw)


# ---------------------------------------------------------------------------------------------
# (e) selection rules, the per-batch overrides and edge shapes
@pytest.mark.parametrize("W,n,nj,maxc,lpw,collide,records", [
    (4096, 10, 0, 0, 4, 32, 32),         # C2: 4096 x stack10
    (65536, 64, 0, 1024, 8, 256, 128),   # C3: 65536 x pile64
    (131072, 20, 19, 0, 4, 32, 32),      # C5: 131072 x legged20 (and the MPC stack)
    (16, 10, 0, 0, 8, 32, 32),           # W <= 16
    (16, 64, 0, 1024, 8, 256, 128),
    (8192, 10, 0, 0, 2, 32, 32),         # stack10 at 8192 worlds
    (8, 40, 0, 0, 8, 128, 128),          # the 40-rock cairn: 780 pairs
])
def test_default_selection(W, n, nj, maxc, lpw, collide, records):
    """Without overrides every batch chooses the documented instances (created, not stepped)."""
    import eggshell_b200 as E
    b = E.Batch(W, n, nj, solver=E.SOLVER_PGS, max_contacts=maxc)
    cfg = b.kernel_config()
    b.close()
    assert cfg == dict(lpw=lpw, worlds_per_warp=32 // lpw, iso=-1, rec_format=-1, run_cap=0, precision=64,
                       collide_threads=collide, records_threads=records), cfg


def test_overrides_are_read_per_batch(monkeypatch):
    """One process, batches created one after the other: each one runs what the environment said
    when it was created."""
    import eggshell_b200 as E
    scene = _scene("stack10", 16)

    def cfg_of(step=False, **kw):
        b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=20, **kw)
        if step:
            b.step(scene["dt"])
        c = b.kernel_config()
        b.close()
        return c

    seen = []
    for v in ("2", "16", None):
        if v is None:
            monkeypatch.delenv("EGG_PGS_LPW")
        else:
            monkeypatch.setenv("EGG_PGS_LPW", v)
        seen.append(cfg_of()["lpw"])
    assert seen == [2, 16, 8], seen
    monkeypatch.setenv("EGG_COLLIDE_NT", "128")
    monkeypatch.setenv("EGG_RECORDS_NT", "64")
    c = cfg_of()
    assert (c["collide_threads"], c["records_threads"]) == (128, 64), c
    monkeypatch.delenv("EGG_COLLIDE_NT")
    monkeypatch.delenv("EGG_RECORDS_NT")
    c = cfg_of()
    assert (c["collide_threads"], c["records_threads"]) == (32, 32), c
    # the run format is decided at the first step: the batch keeps what egg_create read
    monkeypatch.setenv("EGG_PGS_RUNS", "1")
    monkeypatch.setenv("EGG_PGS_RUN_CAP", "1")
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=20)
    monkeypatch.delenv("EGG_PGS_RUNS")
    monkeypatch.delenv("EGG_PGS_RUN_CAP")
    assert cfg_of(step=True)["rec_format"] == 1
    b.step(scene["dt"])
    c = b.kernel_config()
    b.close()
    assert (c["rec_format"], c["run_cap"], c["iso"]) == (2, 1, 2), c
    c = cfg_of(step=True, quirks=RUNS)
    assert c["rec_format"] == 2 and c["run_cap"] == 8, c


@pytest.mark.parametrize("lpw", [1, 16])
def test_edge_shapes_vs_oracle(lpw, monkeypatch):
    """W = 1, W = G - 1 and W = G; a warp group whose worlds have no constraint at all between groups
    that have; one-body worlds (LPW 1)."""
    import eggshell_b200 as E
    G = 32 // lpw
    cases = [("W=1", _cairn_mix(1)), ("W=G", _cairn_mix(G))]
    if G > 1:
        cases.append(("W=G-1", _cairn_mix(G - 1)))
    cases.append(("empty middle group", _cairn_mix(3 * G, lifted=range(G, 2 * G))))
    if lpw == 1:
        for W in (1, 3):
            cases.append((f"one body, W={W}", E.scenes.cairn(W, rocks=1, zb=(0.05, 0.1), seed=44)))
    for what, scene in cases:
        monkeypatch.setenv("EGG_PGS_LPW", str(lpw))
        cfg, sw = _probe(scene, dict(solver=E.SOLVER_PGS))
        assert cfg["lpw"] == lpw, cfg
        worst = stepwise(scene, 3, list(range(scene["W"])), dict(solver=E.SOLVER_PGS), dict(solver=1))
        _report(what, cfg, scene["W"], worst, sw)
