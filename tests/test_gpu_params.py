"""GPU parity beyond the reference's constants: boxes that are not cubes, contact de-duplication and
joint conflicts at larger minimum constraint distances, and every step parameter the C ABI takes per
batch (erp, cfm, tol, gravity, dt, cfm_mode), each against the FP64 oracle one step at a time from
shared state.

`strict_stepwise` is `tests.helpers.stepwise` plus the parts of the step's output that it leaves out:
the whole stats row (stat 7 is reserved and differs by design), the whole status word, the pair-hit
list and the solver residual.  Every case prints the kernel instance it ran, the worst errors, the
sweep range and how often a sweep count was allowed to differ by one at a near-tie.

The scene builders live here; tests/test_param_scenes_oracle.py checks on the CPU that they still
reach what these tests are for (every box-box pair code 1-16, contact-contact de-duplication, joint
conflicts, early exits at a relaxed tolerance)."""
import math

import numpy as np
import pytest

from eggshell_b200 import scenes as S
from tests.helpers import oracle_world, compare_step

pytestmark = pytest.mark.gpu

OVERRIDES = ("EGG_PGS_LPW", "EGG_PGS_MIN_WARPS_PER_SM", "EGG_PGS_RUNS", "EGG_PGS_RUN_CAP", "EGG_PGS_TARGET_CTAS",
             "EGG_COLLIDE_NT", "EGG_RECORDS_NT", "EGG_PGS_ISO")
DENSE, PGS, JACOBI, SOR = 0, 1, 2, 3
RUNS = 3 | 16                   # QUIRKS_REFERENCE | EGG_OPT_PGS_RUNS
CFM_AUTO, CFM_ALWAYS, CFM_NEVER = 0, 1, 2
STATS = ("n_contacts_raw", "n_contacts", "n_rows", "n_pair_hits", "sweeps", "pivots", "cfm_applied")
SIDES = (0.05, 0.1, 0.3, 0.6, 0.9)

# Residual of the solve.  Both sides stopped on the stopping test (residual <= tol): the two residuals
# are sums of |A x - rhs| terms of size tol, computed from |A x| ~ |rhs| ~ 1e2..1e3 with different
# rounding (measured on a B200: up to 0.06 tol at erp = 0.8), so they are compared to within
# RESID_STOP x tol.  Both ran to k_max: within RESID_STOP x tol + RESID_REL x the oracle's residual
# (measured: SOR differs by up to 1.2e-5 x max(residual, tol), the other solvers by < 1e-10).  FP32
# records move A x by ~1e-7 relative and are held to the stopping test only.
RESID_STOP = 0.25
RESID_REL = 1e-6


@pytest.fixture(autouse=True)
def _no_overrides(monkeypatch):
    for k in OVERRIDES:
        monkeypatch.delenv(k, raising=False)


# ---------------------------------------------------------------------------------------------
# Scenes: boxes with three different side lengths.
def box_inertia(m, side):
    """Body-frame inertia of a solid box (body.cc:19-36) for side lengths side[..., 3]."""
    I = np.zeros(side.shape[:-1] + (3, 3))
    sq = side ** 2
    I[..., 0, 0] = m / 12 * (sq[..., 1] + sq[..., 2])
    I[..., 1, 1] = m / 12 * (sq[..., 0] + sq[..., 2])
    I[..., 2, 2] = m / 12 * (sq[..., 0] + sq[..., 1])
    return I


def _with_sides(sc, side, inertia):
    """inertia "box": the box's own anisotropic inertia (M^-1 layout 0); "iso": a sphere-like inertia
    with the mean of its principal moments, different per body (layout 1, which the run format needs)."""
    sc["side"] = np.ascontiguousarray(side, dtype=np.float64)
    I = box_inertia(sc["m"], sc["side"])
    if inertia == "iso":
        I = np.eye(3) * (np.trace(I, axis1=-2, axis2=-1) / 3.0)[..., None, None]
    sc["I"] = I
    return sc


def _blank(W, n, dt=0.005):
    return dict(p=np.zeros((W, n, 3)), R=np.tile(np.eye(3), (W, n, 1, 1)), v=np.zeros((W, n, 3)), w=np.zeros((W, n, 3)),
                m=np.ones((W, n)), I=np.tile(np.eye(3) * 0.015, (W, n, 1, 1)), n=n, W=W, nj=0, dt=dt)


def _rot(axis, a):
    c, s = math.cos(a), math.sin(a)
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    R = np.eye(3)
    R[i, i], R[i, j], R[j, i], R[j, j] = c, -s, s, c
    return R


# exact quarter turns (no rounding in cos / sin): R[:, k] of a box lies exactly on a world axis
QUARTER = [np.eye(3), np.array([[1.0, 0, 0], [0, 0, -1], [0, 1, 0]]), np.array([[0.0, 0, 1], [0, 1, 0], [-1, 0, 0]]),
           np.array([[0.0, -1, 0], [1, 0, 0], [0, 0, 1]])]


def heap(W, n=12, seed=900, inertia="box"):
    """(a) Planks, slabs and rods (every side drawn from SIDES) in a 0.8 m x 0.8 m heap, z in 0.1-0.9 m,
    uniform random orientations, v, w ~ U(+-1)."""
    sc = S.cairn(W, rocks=n, xb=(-0.4, 0.4), yb=(-0.4, 0.4), zb=(0.1, 0.9), seed=seed)
    side = np.random.default_rng(seed + 1).choice(SIDES, size=(W, n, 3))
    sc["m"] = np.ones((W, n))
    sc["name"] = f"heap{n}"
    return _with_sides(sc, side, inertia)


def crosswise(W, layers=6, seed=910, inertia="box"):
    """(b) 0.9 x 0.15 x 0.1 slabs stacked crosswise (every other layer turned by an exact quarter turn),
    each layer's bottom face exactly on the top face of the one below: the face manifolds have depths
    of |depth| <= 1e-9 and aacount = 3, so they are kept whatever their depth (collision.cc:369).
    Odd worlds turn each slab by a small yaw (< 0.02 rad, still aacount >= 2).  The bottom slab is
    1 mm in the ground, so the stack is carried from the first step on: a stack in free fall has
    contacts that carry no load, and their multipliers (~1e-14) sit on the bound of the clamp."""
    rng = np.random.default_rng(seed)
    sc = _blank(W, layers)
    for l in range(layers):
        sc["p"][:, l, 2] = 0.05 + 0.1 * l - 1e-3
        sc["R"][:, l] = QUARTER[3] if l % 2 else np.eye(3)
    sc["p"][:, :, :2] = rng.uniform(-0.02, 0.02, size=(W, layers, 2))
    yaw = rng.uniform(-0.02, 0.02, size=(W, layers))
    yaw[0::2] = 0.0
    sc["R"] = np.einsum("wlij,wljk->wlik", S._rot_z(yaw), sc["R"])
    sc["name"] = "crosswise"
    return _with_sides(sc, np.tile(np.array([0.9, 0.15, 0.1]), (W, layers, 1)), inertia)


# angle between the two crossing rods of world w: near-parallel (edge axis |u_a x u_b| = sin(angle)
# around kTolerance = 1e-9, collision.cc:240) up to crosswise
ROD_ANGLES = (3e-10, 1e-9, 2e-9, 1e-6, 0.02, 0.4, 0.9, 1.4)


def rods(W, seed=920, inertia="box"):
    """(c) Thin rods crossing edge to edge.  Bodies 0 and 1: two 0.9 x 0.05 x 0.05 rods rolled by 45
    degrees about their long axis (diamond cross-section), the upper one turned by ROD_ANGLES[w % 8]
    about z and lowered 1e-4 onto the lower one's top edge.  Bodies 2..5: pick-up sticks (random rods
    and planks, random orientations, crossing each other) dropped 1.5 m away."""
    rng = np.random.default_rng(seed)
    n = 6
    sc = _blank(W, n)
    side = np.zeros((W, n, 3))
    side[:, :2] = (0.9, 0.05, 0.05)
    h = 0.05 * math.sqrt(0.5)                      # half the diagonal of the cross-section
    roll = _rot(0, math.pi / 4)
    for w in range(W):
        a = ROD_ANGLES[w % len(ROD_ANGLES)]
        sc["R"][w, 0] = roll
        sc["R"][w, 1] = _rot(2, a) @ roll
        sc["p"][w, 0] = (0.0, 0.0, h - 1e-3)
        sc["p"][w, 1] = (0.0, 0.0, 3 * h - 1e-3 - 1e-4)
    side[:, 2:] = rng.choice([(0.9, 0.05, 0.05), (0.6, 0.1, 0.05), (0.9, 0.1, 0.1), (0.6, 0.05, 0.1)], size=(W, n - 2))
    q = rng.normal(size=(W, n - 2, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    sc["R"][:, 2:] = S.quat_to_mat(q)
    sc["p"][:, 2:, 0] = 1.5 + rng.uniform(-0.1, 0.1, size=(W, n - 2))
    sc["p"][:, 2:, 1] = rng.uniform(-0.1, 0.1, size=(W, n - 2))
    sc["p"][:, 2:, 2] = 0.04 + 0.06 * np.arange(n - 2) + rng.uniform(0, 0.01, size=(W, n - 2))
    sc["v"][:, 2:] = rng.uniform(-0.3, 0.3, size=(W, n - 2, 3))
    sc["name"] = "rods"
    return _with_sides(sc, side, inertia)


def ground(W, seed=930, inertia="box"):
    """(d) One 0.6 x 0.1 x 0.3 box per world (the side lengths permuted per world) resting on the
    ground in a different orientation: flat on each face (exact quarter turns), on an edge, on a
    vertex, at random; its lowest vertex 1e-3 below the ground."""
    rng = np.random.default_rng(seed)
    sc = _blank(W, 1)
    perms = [(0, 1, 2), (1, 2, 0), (2, 0, 1), (0, 2, 1)]
    side = np.zeros((W, 1, 3))
    for w in range(W):
        side[w, 0] = np.array([0.6, 0.1, 0.3])[list(perms[w % 4])]
        k = w % 6
        if k < 3:
            R = QUARTER[k + 1] if k else np.eye(3)
        elif k == 3:
            R = _rot(0, math.pi / 4 + 0.01 * w)
        elif k == 4:
            R = _rot(1, 0.6155) @ _rot(0, math.pi / 4)
        else:
            q = rng.normal(size=4)
            R = S.quat_to_mat(q / np.linalg.norm(q))
        sc["R"][w, 0] = R
        corners = np.array([[x, y, z] for x in (-.5, .5) for y in (-.5, .5) for z in (-.5, .5)]) * side[w, 0]
        sc["p"][w, 0] = (0.1 * w, 0.0, -(corners @ R.T)[:, 2].min() - 1e-3)
    sc["v"][:, 0] = rng.uniform(-0.05, 0.05, size=(W, 3))
    sc["w"][:, 0] = rng.uniform(-0.2, 0.2, size=(W, 3))
    sc["name"] = "ground"
    return _with_sides(sc, side, inertia)


BOX_SCENES = {"heap": (heap, 16, 4), "crosswise": (crosswise, 8, 5), "rods": (rods, 8, 5), "ground": (ground, 12, 6)}


def coincident_chain(W, links=5):
    """A hanging chain (bodies as scenes.chain) with one more ball joint between links 1 and 2: on even
    worlds at the same anchors as the chain's own joint between them (the two joints coincide: the
    reference Panics, the step raises EGG_ST_JOINT_CONFLICT), on odd worlds 0.02 m along the links'
    x axis (no conflict at the default distance)."""
    sc = S.chain(W, links=links, anchor=(0.0, 0.0, 2.0))
    shift = np.where(np.arange(W)[:, None] % 2 == 1, np.array([0.02, 0.0, 0.0]), 0.0)
    sc["i0"] = np.append(sc["i0"], np.int32(1)).astype(np.int32)
    sc["i1"] = np.append(sc["i1"], np.int32(2)).astype(np.int32)
    sc["c0"] = np.concatenate([sc["c0"], (sc["c0"][:, 1] + shift)[:, None]], axis=1)
    sc["c1"] = np.concatenate([sc["c1"], (sc["c1"][:, 1] + shift)[:, None]], axis=1)
    sc["nj"] = links + 1
    sc["name"] = "coincident chain"
    return sc


def rocks(W=8, seed=21):
    """Contact scene of the parameter cases: four cubes falling onto the ground and onto each other."""
    return S.cairn(W, rocks=4, zb=(0.15, 0.45), seed=seed)


def low_chain(W=2):
    """Jointed scene of the dense parameter cases: a 6-link chain anchored just above the ground."""
    return S.chain(W, links=6, anchor=(0.0, 0.0, 0.25), seed=5, anchor_jitter=0.05)


def one_vertex_boxes(mus, seed=77):
    """Two boxes apart from each other, each resting on exactly one vertex (3 rows each, a full-rank
    system), the second heavier by mu: cond(A) grows with mu (test_gpu_parity.test_cfm_decision_sweep)."""
    q = np.random.default_rng(seed).normal(size=(2, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    Rm = S.quat_to_mat(q)
    sc = S.cairn(len(mus), rocks=2, seed=5)
    sc["R"][:] = Rm[None]
    sc["v"][:] = 0.0
    sc["w"][:] = 0.0
    corners = np.array([[sx, sy, sz] for sx in (-.15, .15) for sy in (-.15, .15) for sz in (-.15, .15)])
    for k in range(2):
        low = np.sort((corners @ Rm[k].T)[:, 2])
        assert low[1] - low[0] > 5e-3
        sc["p"][:, k, :] = (2.0 * k, 0.0, -low[0] - 1e-3)
    sc["m"][:, 1] = mus
    sc["I"][:, 1] = np.eye(3)[None] * (0.1 * np.asarray(mus))[:, None, None]
    sc["name"] = "one-vertex boxes"
    return sc


def sub_scene(scene, pick):
    """The worlds `pick` of a scene as a scene of their own."""
    W = scene["W"]
    sub = dict(scene)
    for key, val in scene.items():
        if isinstance(val, np.ndarray) and val.shape[:1] == (W,):
            sub[key] = val[pick].copy()
    sub["W"] = len(pick)
    return sub


# ---------------------------------------------------------------------------------------------
# The strict per-step comparison.
def split_kw(solver, **p):
    """Batch and oracle keyword arguments of one parameter set (the oracle has no opt-in quirks)."""
    bkw, okw = dict(solver=solver), dict(solver=solver)
    for k, v in p.items():
        if k == "min_dist":
            bkw["min_constraint_dist"] = v
            okw["min_dist"] = v
        elif k == "quirks":
            bkw[k] = v
            okw[k] = v & 3
        elif k == "precision":
            bkw[k] = v
        else:
            bkw[k] = v
            okw[k] = v
    return bkw, okw


def kernel_name(cfg, solver):
    if solver == DENSE:
        return "egg_dense (Schur + Murty)"
    if solver in (JACOBI, SOR):
        return "egg_iter_kernel " + ("Jacobi" if solver == JACOBI else "SOR")
    if cfg["rec_format"] == 2:
        return f"egg_pgs_runs_kernel<{cfg['lpw']},{cfg['iso']}>"
    return f"egg_pgs_stream_kernel<{cfg['lpw']},{8 if cfg['iso'] == 0 else 12},{cfg['iso']},{str(cfg['precision'] == 32).lower()}>"


def strict_stepwise(scene, nsteps, solver, idx=None, state_tol=None, lam_tol=1e-9, slack=False, what="", **params):
    """One step at a time from shared state against the oracle at the parameters `params` (oracle
    names: erp, cfm, tol, k_max, gravity, min_dist, cfm_mode, quirks; plus precision = 32).

    Per step and world: contacts, state and multipliers as compare_step, within state_tol (default
    1e-9; FP32 records: 1e-4, no multipliers) and lam_tol; the whole stats row but stat 7 and the whole status word equal to the
    oracle's; the pair-hit list (i, j, code, contacts before de-duplication) bit-exact; clamp states
    bit-exact (FP64); the residual as RESID_STOP and RESID_REL say; the near-tie probe of
    tests.helpers.stepwise (PGS, FP64).  slack: a sweep count may differ by one where the oracle shows
    why (tests.helpers.stepwise_fp32(sweep_slack=True)); that world's state is not compared on that
    step.  Returns (worst errors and counts, kernel config, per-step oracle stats)."""
    import eggshell_b200 as E
    fp32 = params.get("precision", 64) == 32
    tol = (1e-4 if fp32 else 1e-9) if state_tol is None else state_tol
    slack = slack or fp32
    bkw, okw = split_kw(solver, **params)
    stop, k_max = okw.get("tol", 1e-9), okw.get("k_max", 500)
    idx = list(range(scene["W"])) if idx is None else list(idx)
    b = E.scenes.make_batch(scene, taps=True, **bkw)
    ows = [oracle_world(scene, wi, **okw)[0] for wi in idx]
    dt = scene["dt"]
    worst = dict(near_tie=0, exact_sweep_plus_one=0, resid_stop=0.0, resid_kmax=0.0, sweeps_min=1 << 30, sweeps_max=0)
    history = []
    cfg = None
    for s in range(nsteps):
        p, R, v, w = b.bodies()
        for k, wi in enumerate(idx):
            ows[k].set_state(p[wi], R[wi], v[wi], w[wi])
        b.step(dt)
        for ow in ows:
            ow.step(dt)
        if cfg is None:
            cfg = b.kernel_config()
        st, ph, con = b.status(), b.pair_hits(), b.contacts()
        ostats = [ow.stats() for ow in ows]
        history.append(ostats)
        tie = set()
        for k, wi in enumerate(idx):
            os_ = ostats[k]
            kg, ko = int(st["sweeps"][wi]), os_["sweeps"]
            worst["sweeps_min"] = min(worst["sweeps_min"], kg)
            worst["sweeps_max"] = max(worst["sweeps_max"], kg)
            if kg != ko:
                assert slack and abs(kg - ko) == 1, f"{what} step {s} world {wi}: sweeps {kg} != {ko} (oracle residual {os_['residual']:.3e})"
                tie.add(k)
                if fp32 and kg == ko + 1 and os_["residual"] < 1e-11:
                    worst["exact_sweep_plus_one"] += 1       # the oracle's last sweep was exact (stepwise_fp32)
                    continue
                ow2 = oracle_world(scene, wi, **dict(okw, k_max=min(kg, ko)))[0]
                ow2.set_state(p[wi], R[wi], v[wi], w[wi])
                ow2.step(dt)
                r = ow2.stats()["residual"]
                assert abs(r / stop - 1.0) < 1e-3, f"{what} step {s} world {wi}: sweeps {kg} != {ko}, oracle residual {r:.6e} at sweep {min(kg, ko)} is no near-tie"
                worst["near_tie"] += 1
        keep = [k for k in range(len(idx)) if k not in tie]
        e = compare_step(b, [ows[k] for k in keep], [idx[k] for k in keep], tol=tol, check_lambda=not fp32, lam_tol=lam_tol)
        for key, val in e.items():
            worst[key] = max(worst.get(key, 0.0), val)
        for k, wi in enumerate(idx):
            os_ = ostats[k]
            for key in STATS:
                if key == "sweeps" and k in tie:
                    continue
                assert st[key][wi] == os_[key], f"{what} step {s} world {wi}: {key} {st[key][wi]} != oracle {os_[key]}"
            assert st["status"][wi] == os_["status"], f"{what} step {s} world {wi}: status {st['status'][wi]} != oracle {os_['status']}"
            oh = ows[k].pair_hits()
            nh = int(ph["n"][wi])
            assert nh == len(oh["i"]), f"{what} step {s} world {wi}: {nh} pair hits != oracle {len(oh['i'])}"
            for key in ("i", "j", "code", "count"):
                assert np.array_equal(ph[key][wi, :nh], oh[key]), f"{what} step {s} world {wi}: pair-hit {key} differs"
            rg, ro = float(st["residual"][wi]), os_["residual"]
            if solver == DENSE:
                assert rg == 0.0 and ro == 0.0
            elif k not in tie:
                if os_["sweeps"] < k_max:            # stopped on the stopping test (or had no rows)
                    assert rg <= stop and ro <= stop, f"{what} step {s} world {wi}: residual {rg:.3e} / oracle {ro:.3e} above tol {stop:g}"
                    if not fp32:
                        worst["resid_stop"] = max(worst["resid_stop"], abs(rg - ro) / stop)
                elif not fp32:
                    worst["resid_kmax"] = max(worst["resid_kmax"], abs(rg - ro) / (RESID_STOP * stop + RESID_REL * ro))
            if fp32 or k in tie:
                continue
            lam, rhs, rs = ows[k].solution()
            lam, rs = np.asarray(lam), np.asarray(rs)
            assert np.array_equal(con["row_state"][wi, :len(rs)], rs), f"{what} step {s} world {wi}: row clamp states differ"
            if solver != PGS:
                continue
            # near-tie probe of tests.helpers.stepwise: equal clamp states only mean something if no free
            # multiplier sits within rounding distance of a bound (q2: the first contact block after the
            # joints is projected with the joint's bounds)
            blk = np.arange(len(lam)) // 3
            bounded = (blk > scene["nj"]) if scene["nj"] else np.ones(len(lam), dtype=bool)
            free = (rs == 0) & bounded
            if free.any() and os_["sweeps"] > 0:
                row = np.arange(len(lam)) % 3
                dist = np.where(row < 2, 1.0 - np.abs(lam), np.abs(lam))[free]
                diff = float(np.max(np.abs(con["lam"][wi, :len(lam)] - lam)))
                worst["clamp_margin_over_diff"] = min(worst.get("clamp_margin_over_diff", np.inf), float(dist.min()) / max(diff, 1e-300))
        assert worst["resid_stop"] <= RESID_STOP, f"{what}: residuals at the stopping test differ by {worst['resid_stop']:.3e} x tol"
        assert worst["resid_kmax"] <= 1.0, f"{what}: residuals at k_max differ by {worst['resid_kmax']:.3e} x the allowed difference"
    b.close()
    if "clamp_margin_over_diff" in worst:
        assert worst["clamp_margin_over_diff"] > 10.0, f"{what}: near-tie: a free multiplier is within 10x of the CUDA-vs-oracle difference of its bound"
    errs = " ".join(f"{k} {worst[k]:.1e}" for k in ("p", "R", "v", "w", "lam", "geom") if k in worst)
    print(f"{what}: {kernel_name(cfg, solver)} | {len(idx)} worlds x {nsteps} steps | {errs} | residual {worst['resid_stop']:.1e} x tol "
          f"at the test, {worst['resid_kmax']:.1e} of the allowed at k_max | sweeps {worst['sweeps_min']}/{worst['sweeps_max']} | "
          f"near ties {worst['near_tie']}, exact sweep + 1 {worst['exact_sweep_plus_one']}")
    return worst, cfg, history


# ---------------------------------------------------------------------------------------------
# 2. Boxes that are not cubes.
@pytest.mark.parametrize("name", list(BOX_SCENES))
@pytest.mark.parametrize("variant", ["default", "lpw1", "lpw16", "fp32", "runs"])
def test_box_scene_vs_oracle(name, variant, monkeypatch):
    """The four box scenes through the PGS stream kernel at its default instance, at 1 and 16 lanes per
    world, with FP32 records, and through the run format (isotropic inertia, which it needs)."""
    build, W, steps = BOX_SCENES[name]
    scene = build(W, inertia="iso" if variant == "runs" else "box")
    kw = dict(k_max=500)
    if variant.startswith("lpw"):
        monkeypatch.setenv("EGG_PGS_LPW", variant[3:])
    if variant == "fp32":
        kw["precision"] = 32
    if variant == "runs":
        kw["quirks"] = RUNS
    worst, cfg, hist = strict_stepwise(scene, steps, PGS, what=f"{name} {variant}", **kw)
    assert (cfg["iso"] >= 1) if variant == "runs" else (cfg["iso"] == 0), cfg
    assert cfg["rec_format"] == (2 if variant == "runs" else 1), cfg
    if variant.startswith("lpw"):
        assert cfg["lpw"] == int(variant[3:]), cfg
    assert sum(o["n_contacts"] for step in hist for o in step) > 0


@pytest.mark.parametrize("name,W,n,steps", [("ground", 12, 1, 6), ("heap", 6, 4, 5)])
def test_box_scene_dense_vs_oracle(name, W, n, steps):
    """The dense path on the one-box worlds and on a heap of four boxes."""
    scene = ground(W) if name == "ground" else heap(W, n=n, seed=940)
    worst, cfg, hist = strict_stepwise(scene, steps, DENSE, what=f"{name} dense")
    assert sum(o["pivots"] for step in hist for o in step) > 0


def test_sides_through_set_bodies_and_set_shapes_are_the_same():
    """Box side lengths handed to egg_set_bodies(side) and to egg_set_shapes(0, dims) give the same bits:
    contacts, pair hits, multipliers and state over three steps of the heap."""
    import eggshell_b200 as E
    scene = heap(8)
    as_shapes = dict(scene)
    del as_shapes["side"]
    as_shapes["shape"] = np.zeros((8, scene["n"]), dtype=np.int32)
    as_shapes["dims"] = scene["side"]
    out = []
    for sc in (scene, as_shapes):
        b = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, k_max=50, taps=True)
        b.step(sc["dt"], n_steps=3)
        res = dict(b.contacts())
        res.update({"hit_" + k: v for k, v in b.pair_hits().items()})
        res.update(zip("pRvw", b.bodies()))
        out.append(res)
        b.close()
    for key in out[0]:
        assert np.array_equal(out[0][key], out[1][key]), key
    assert int(out[0]["hit_n"].sum()) > 0


def test_box_heap_collide_instances_are_bit_identical(monkeypatch):
    """Forced narrowphase threads per world {32, 64, 128, 256} give the same contacts, pair hits and
    state bit for bit on the heap (test_pgs_instances.test_presolve_instances_are_bit_identical for
    cubes)."""
    import eggshell_b200 as E
    scene = heap(8)
    ref = None
    for nt in (None, 32, 64, 128, 256):
        if nt is None:
            monkeypatch.delenv("EGG_COLLIDE_NT", raising=False)
        else:
            monkeypatch.setenv("EGG_COLLIDE_NT", str(nt))
        b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=20, taps=True)
        b.step(scene["dt"], n_steps=2)
        cfg = b.kernel_config()
        assert int(np.bitwise_or.reduce(b.status()["status"])) == 0
        out = dict(b.contacts())
        out.update({"hit_" + k: v for k, v in b.pair_hits().items()})
        out.update(zip("pRvw", b.bodies()))
        b.close()
        if nt is not None:
            assert cfg["collide_threads"] == nt, cfg
        if ref is None:
            ref, dflt = out, cfg["collide_threads"]
            continue
        for key, a in out.items():
            assert np.array_equal(a, ref[key]), f"EGG_COLLIDE_NT={nt}: {key} differs from the default ({dflt} threads)"
    print(f"heap: egg_collide_kernel<32|64|128|256> bit-identical to the default <{dflt}>, {int(ref['count'].sum())} contacts, "
          f"{int(ref['hit_n'].sum())} pair hits")


def test_full_size_heap_worlds_are_independent_of_the_batch(monkeypatch):
    """65536 heaps at K = 10: no status flag, finite state; sampled worlds (first, middle and last
    groups) stepped again in a batch of their own at another lane count give the same bits, and that
    batch matches the oracle (test_gpu_parity.test_full_size_worlds_are_independent_of_the_batch)."""
    import eggshell_b200 as E
    W, k_max = 65536, 10
    scene = heap(W)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max)
    b.step(scene["dt"])
    big = [x.copy() for x in b.bodies()]
    st_big = b.status()
    big_lpw = b.kernel_config()["lpw"]
    assert int(np.bitwise_or.reduce(st_big["status"])) == 0, np.unique(st_big["status"]).tolist()
    assert all(np.isfinite(x).all() for x in big)
    assert int(st_big["n_contacts"].min()) > 0
    b.close()
    pick = np.array([0, 1, 5, W // 3, W // 2 + 3, W - 34, W - 2, W - 1])
    sub = sub_scene(scene, pick)
    small_lpw = 16 if big_lpw != 16 else 2
    monkeypatch.setenv("EGG_PGS_LPW", str(small_lpw))
    sb = E.scenes.make_batch(sub, solver=E.SOLVER_PGS, k_max=k_max, taps=True)
    assert sb.kernel_config()["lpw"] == small_lpw
    ows = [oracle_world(sub, k, solver=1, k_max=k_max)[0] for k in range(len(pick))]
    sb.step(sub["dt"])
    for ow in ows:
        ow.step(sub["dt"])
    st_small = sb.status()
    for a, c in zip(sb.bodies(), big):
        assert np.array_equal(a.view(np.uint64), c[pick].view(np.uint64)), "heap: a world's step depends on its batch"
    for key in STATS:
        assert np.array_equal(st_small[key], st_big[key][pick]), key
    worst = compare_step(sb, ows, list(range(len(pick))))
    for k, ow in enumerate(ows):
        assert st_small["cfm_applied"][k] == ow.stats()["cfm_applied"] and st_small["status"][k] == ow.stats()["status"]
    print(f"heap x {W} (LPW {big_lpw}) vs {len(pick)} of them (LPW {small_lpw}): same bits; vs oracle {worst}")
    sb.close()


# ---------------------------------------------------------------------------------------------
# 3. De-duplication and joint conflicts.
def _dedup_scene(name):
    if name == "stack10":
        return S.stack10(4, seed=1000), 3, dict(k_max=100)
    if name == "pile64":
        return S.pile64(2, seed=3000), 2, dict(k_max=50)
    if name == "cairn":
        return S.cairn(8, rocks=4, zb=(0.2, 1.0), seed=11), 12, {}
    if name == "chain32":
        return S.chain32(2, seed=4000), 3, dict(k_max=100)
    return heap(8), 3, dict(k_max=100)


@pytest.mark.parametrize("name,dmin,solver", [
    ("stack10", 0.03, PGS), ("stack10", 0.1, PGS), ("pile64", 0.03, PGS), ("pile64", 0.1, PGS),
    ("cairn", 0.03, PGS), ("cairn", 0.1, PGS), ("chain32", 0.03, PGS), ("chain32", 0.1, PGS),
    ("chain32", 0.03, DENSE), ("chain32", 0.1, DENSE), ("heap", 0.03, PGS),
    ("stack10", 0.0, PGS), ("heap", 0.0, PGS), ("chain32", 0.0, DENSE)])
def test_dedup_distance_vs_oracle(name, dmin, solver):
    """min_constraint_dist well above the default 1e-6: contacts of one body pair closer than it are
    dropped (the later one) and contacts closer than it to a joint of that pair go; the raw and kept
    counts, the kept list and everything downstream equal to the oracle's.  At 0 nothing is dropped."""
    scene, steps, kw = _dedup_scene(name)
    if solver == DENSE:
        kw = {}
    worst, cfg, hist = strict_stepwise(scene, steps, solver, min_dist=dmin, what=f"{name} min_dist {dmin:g}", **kw)
    dropped = sum(o["n_contacts_raw"] - o["n_contacts"] for step in hist for o in step)
    raw = sum(o["n_contacts_raw"] for step in hist for o in step)
    print(f"  {name} min_dist {dmin:g}: {dropped} of {raw} contacts dropped by de-duplication")
    if dmin == 0.0:
        assert dropped == 0
    else:
        assert dropped > 0


def test_joint_conflict_vs_oracle():
    """EGG_ST_JOINT_CONFLICT on exactly the worlds where the oracle raises it, sticky from egg_init on:
    the hinge of scenes.rounds (two ball joints 0.2 m apart) at min_constraint_dist 0.25, and a chain
    whose even worlds carry two coincident ball joints (odd worlds: 0.02 m apart, default distance)."""
    import eggshell_b200 as E
    sc = S.rounds(4)
    worst, cfg, hist = strict_stepwise(sc, 4, PGS, k_max=100, min_dist=0.25, lam_tol=1e-8, what="rounds min_dist 0.25")
    assert all(o["status"] & 2 for step in hist for o in step)
    for solver in (PGS, DENSE):
        sc = coincident_chain(6)
        b = E.scenes.make_batch(sc, solver=solver)
        st0 = b.status()["status"].copy()
        b.close()
        expect = (np.arange(6) % 2 == 0)
        assert np.array_equal((st0 & 2) != 0, expect), st0
        worst, cfg, hist = strict_stepwise(sc, 4, solver, k_max=100, what=f"coincident chain solver {solver}")
        for step in hist:
            assert np.array_equal(np.array([(o["status"] & 2) != 0 for o in step]), expect)


# ---------------------------------------------------------------------------------------------
# 4. Step parameters.
def _legged(W=4):
    return S.legged20(W, seed=5000)


def tol_cases(solver):
    """(scene, steps) of test_tol_vs_oracle.  Jacobi is not a contraction on the legged tree: on the
    oracle, six sweeps turn a 1e-15 change of the state into 2e-9 by the third step, so it runs the two
    steps of test_gpu_parity.test_jacobi_sor_stepwise there."""
    return [(rocks(), 10), (_legged(2), 2) if solver == JACOBI else (_legged(4), 3)]


@pytest.mark.parametrize("erp", [0.0, 0.8])
def test_erp_vs_oracle(erp):
    """erp scales the position error in the record rhs (egg_record.cuh) and in the dense rhs."""
    strict_stepwise(rocks(), 10, PGS, erp=erp, what=f"rocks erp {erp}")
    strict_stepwise(_legged(), 3, PGS, erp=erp, k_max=100, what=f"legged20 erp {erp}")
    strict_stepwise(rocks(4), 10, DENSE, erp=erp, what=f"rocks dense erp {erp}")
    strict_stepwise(low_chain(), 5, DENSE, erp=erp, what=f"chain dense erp {erp}")


@pytest.mark.parametrize("cfm", [1e-4, 0.1])
def test_cfm_vs_oracle(cfm):
    """cfm reaches 1/(D + cfm) of the records (FP64 and FP32), the residual rhs - A x - cfm x of every
    matrix-free solver, and the dense diagonal when the condition test adds it."""
    strict_stepwise(rocks(), 10, PGS, cfm=cfm, what=f"rocks cfm {cfm}")
    strict_stepwise(_legged(), 3, PGS, cfm=cfm, k_max=100, what=f"legged20 cfm {cfm}")
    strict_stepwise(rocks(), 10, PGS, cfm=cfm, precision=32, what=f"rocks FP32 cfm {cfm}")
    strict_stepwise(_legged(), 3, PGS, cfm=cfm, k_max=100, precision=32, what=f"legged20 FP32 cfm {cfm}")
    _, _, hist = strict_stepwise(rocks(4), 10, DENSE, cfm=cfm, what=f"rocks dense cfm {cfm}")
    _, _, hist2 = strict_stepwise(low_chain(), 5, DENSE, cfm=cfm, what=f"chain dense cfm {cfm}")
    assert any(o["cfm_applied"] for step in hist + hist2 for o in step)
    # Jacobi is not a contraction on these systems: a few sweeps (test_gpu_parity.test_jacobi_sor_stepwise)
    for solver, km in ((JACOBI, 6), (SOR, 40)):
        strict_stepwise(rocks(), 8, solver, cfm=cfm, k_max=km, what=f"rocks {'jacobi' if solver == JACOBI else 'sor'} cfm {cfm}")
        strict_stepwise(_legged(2), 2, solver, cfm=cfm, k_max=km, what=f"legged20 {'jacobi' if solver == JACOBI else 'sor'} cfm {cfm}")


def test_cfm_zero_on_well_posed_scenes():
    """cfm = 0 with PGS where A is nonsingular: a hanging chain (joint rows only) and boxes resting on
    one vertex each; cfm_applied is 0 on both sides."""
    chain = S.chain(4, links=6, anchor=(0.0, 0.0, 3.0), seed=3, v_jitter=0.2)
    _, _, hist = strict_stepwise(chain, 4, PGS, cfm=0.0, k_max=200, what="hanging chain cfm 0")
    _, _, hist2 = strict_stepwise(one_vertex_boxes([1.0, 3.0, 10.0]), 3, PGS, cfm=0.0, what="one-vertex boxes cfm 0")
    assert not any(o["cfm_applied"] for step in hist + hist2 for o in step)
    assert all(o["n_rows"] > 0 for step in hist for o in step)


@pytest.mark.parametrize("tol", [1e-6, 1e-3])
@pytest.mark.parametrize("variant", ["lpw1", "lpw16", "runs", "jacobi", "sor"])
def test_tol_vs_oracle(tol, variant, monkeypatch):
    """A relaxed stopping tolerance: the probe's lower bound and the exact residual decide the exit
    (stream kernel at 1 and 16 lanes per world, run format, Jacobi / SOR); at least one world of each
    case exits before k_max."""
    solver = {"jacobi": JACOBI, "sor": SOR}.get(variant, PGS)
    kw = dict(tol=tol, cfm=0.1)
    if variant.startswith("lpw"):
        monkeypatch.setenv("EGG_PGS_LPW", variant[3:])
    if variant == "runs":
        kw["quirks"] = RUNS
    kw["k_max"] = {JACOBI: 6, SOR: 40}.get(solver, 500)
    early = 0
    for sc, steps in tol_cases(solver):
        _, cfg, hist = strict_stepwise(sc, steps, solver, slack=True, what=f"{sc['name']} {variant} tol {tol:g}", **kw)
        early += sum(0 < o["sweeps"] < kw["k_max"] for step in hist for o in step)
        if variant.startswith("lpw"):
            assert cfg["lpw"] == int(variant[3:]), cfg
        if variant == "runs":
            assert cfg["rec_format"] == 2, cfg
    assert early > 0, "no world exited early"


@pytest.mark.parametrize("gravity", [(1.5, -2.0, -9.8), (0.0, 0.0, -20.0)])
def test_gravity_vs_oracle(gravity):
    """Gravity enters f_ext at egg_init; tilted, it drives the friction rows to their bounds."""
    sat = 0
    for sc, steps, solver in ((rocks(), 10, PGS), (low_chain(4), 4, PGS), (rocks(4), 10, DENSE), (low_chain(2), 4, DENSE)):
        b_kw = dict(k_max=200) if solver == PGS else {}
        worst, cfg, hist = strict_stepwise(sc, steps, solver, gravity=gravity, what=f"{sc['name']} solver {solver} gravity {gravity}", **b_kw)
        if solver == PGS:
            ow = oracle_world(sc, 0, solver=1, gravity=gravity)[0]
            for _ in range(steps):
                ow.step(sc["dt"])
                lam, rhs, rs = ow.solution()
                rs = np.asarray(rs)
                row = np.arange(len(rs)) % 3
                sat += int(np.sum(((rs == 1) | (rs == 2)) & (row < 2) & (np.arange(len(rs)) // 3 >= sc["nj"])))
    if gravity[0] != 0.0:
        assert sat > 0, "no friction row reached its bound"


@pytest.mark.parametrize("dt", [0.02, 1.0 / 60.0])
def test_dt_vs_oracle(dt):
    """A coarser time step: rhs = -erp/dt^2 err - J (v/dt + M^-1 f), positions and orientations."""
    for sc, steps, solver in ((rocks(), 8, PGS), (_legged(4), 3, PGS), (rocks(4), 8, DENSE), (low_chain(2), 4, DENSE)):
        sc["dt"] = dt
        kw = dict(k_max=100) if sc["name"] == "legged20" else {}
        strict_stepwise(sc, steps, solver, what=f"{sc['name']} solver {solver} dt {dt:.4g}", **kw)


def _mu_star():
    """The mass ratio at which the oracle's condition number of A crosses 1e7 (bisection)."""
    from oracle import pyoracle as O
    lo, hi = 1e5, 1e9
    for _ in range(40):
        mid = math.sqrt(lo * hi)
        ow = oracle_world(one_vertex_boxes([mid]), 0, solver=0)[0]
        ow.update_contacts()
        if O.condition_number(ow.dense_A(0.0)) < 1e7:
            lo = mid
        else:
            hi = mid
    return math.sqrt(lo * hi)


def test_cfm_mode_vs_oracle():
    """The dense path's cfm decision bypass: CFM_ALWAYS on worlds where AUTO adds no cfm, CFM_NEVER on
    full-rank worlds where AUTO adds it.  cfm_applied must differ from AUTO's decision on every world.

    CFM_NEVER solves A x = b with cond(A) up to ~1e9 and no regularisation.  Two backward-stable
    solvers (the device's LDL^T-based Murty steps, the oracle's) agree only to about cond(A) x eps
    relative, so the multipliers and the state are held to max(1e-9, 100 cond(A) eps) with cond(A) the
    oracle's condition number of the worlds' A (2.2e-5 at cond 1e9; measured on a B200: 5e-16)."""
    from oracle import pyoracle as O
    mu = _mu_star()
    low = one_vertex_boxes(mu * np.array([1e-3, 1e-2, 0.1, 0.5]))
    high = one_vertex_boxes(mu * np.array([9.0, 30.0, 99.0]))
    for sc, mode, auto in ((low, CFM_ALWAYS, 0), (high, CFM_NEVER, 1)):
        _, _, hist = strict_stepwise(sc, 1, DENSE, what=f"one-vertex boxes AUTO (expect {auto})")
        assert all(o["cfm_applied"] == auto for o in hist[0]), [o["cfm_applied"] for o in hist[0]]
        conds = []
        for w in range(sc["W"]):
            ow = oracle_world(sc, w, solver=0)[0]
            ow.update_contacts()
            conds.append(O.condition_number(ow.dense_A(0.0)))
        t = max(1e-9, 100 * max(conds) * np.finfo(float).eps) if mode == CFM_NEVER else 1e-9
        _, _, hist = strict_stepwise(sc, 3, DENSE, cfm_mode=mode, state_tol=t, lam_tol=t,
                                     what=f"one-vertex boxes cfm_mode {mode} (cond <= {max(conds):.2e}, tol {t:.1e})")
        assert all(o["cfm_applied"] == 1 - auto for step in hist for o in step)
