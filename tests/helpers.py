"""Shared helpers for the parity tests: build CPU-oracle worlds from the same scene arrays that
feed the GPU batch, and compare one step at a time from shared state (BASELINE.json north_star)."""
import numpy as np

from oracle import pyoracle as O


def oracle_world(scene, w, **params):
    W = O.World()
    W.set_bodies(scene["p"][w], scene["R"][w], scene["v"][w], scene["w"][w], scene["m"][w], scene["I"][w],
                 None if "side" not in scene else scene["side"][w])
    if "shape" in scene:
        W.set_shapes(scene["shape"][w], scene["dims"][w])
    if scene["nj"]:
        W.set_joints(scene["i0"], scene["i1"], scene["c0"][w], scene["c1"][w])
    W.set_params(**params)
    st = W.init()
    if "f_ext" in scene:
        W.set_fext(scene["f_ext"][w])
    return W, st


# Natural scale of every compared field: an error is relative to max(|reference|_inf, scale), so a
# field that happens to be near zero in one world is judged against the size it has in the scene,
# not against 1.0.  Lengths: the cube side (body.h:91); velocities: what gravity adds in the
# shortest time step used by any scene (9.8 x 1e-3, constants.h:6-8); angular velocities: the same
# over one cube side; multipliers: the weight of one body (rows are acceleration-level,
# ensembles.cc:569-570).
SCALE = dict(p=0.3, R=1.0, v=9.8e-3, w=9.8e-3 / 0.3, lam=9.8, pos=0.3, nrm=1.0, depth=0.3, resid=1e-3)


def rel_err(a, b, floor):
    """max |a-b| / max(|b|_inf, floor); `floor` is the field's natural scale (SCALE[...])."""
    a, b = np.asarray(a), np.asarray(b)
    if a.size == 0:
        return 0.0
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), floor))


def compare_step(batch, worlds, scene_W_indices, tol=1e-9, check_lambda=True, lam_tol=None):
    """After both sides stepped once from the same state: discrete outputs bit-exact, state and
    multipliers within `tol` relative (north_star: 1e-9 in FP64).  Returns a dict of worst errors."""
    p, R, v, w = batch.bodies()
    con = batch.contacts()
    st = batch.status()
    worst = dict(p=0.0, R=0.0, v=0.0, w=0.0, lam=0.0, geom=0.0)
    for k, wi in enumerate(scene_W_indices):
        ow = worlds[k]
        op, oR, ov, owv = ow.bodies()
        oc = ow.contacts()
        os_ = ow.stats()
        nc = os_["n_contacts"]
        assert con["count"][wi] == nc, f"world {wi}: contact count {con['count'][wi]} != oracle {nc}"
        assert st["n_contacts_raw"][wi] == os_["n_contacts_raw"], f"world {wi}: raw contact count"
        assert st["n_pair_hits"][wi] == os_["n_pair_hits"], f"world {wi}: colliding pair count"
        assert np.array_equal(con["i0"][wi, :nc], oc["i0"]) and np.array_equal(con["i1"][wi, :nc], oc["i1"]), \
            f"world {wi}: contact body indices / order differ"
        assert np.array_equal(con["code"][wi, :nc], oc["code"]), f"world {wi}: collision codes differ"
        worst["geom"] = max(worst["geom"], rel_err(con["pos"][wi, :nc], oc["pos"], SCALE["pos"]),
                            rel_err(con["nrm"][wi, :nc], oc["nrm"], SCALE["nrm"]),
                            rel_err(con["depth"][wi, :nc], oc["depth"], SCALE["depth"]))
        worst["p"] = max(worst["p"], rel_err(p[wi], op, SCALE["p"]))
        worst["R"] = max(worst["R"], rel_err(R[wi], oR, SCALE["R"]))
        worst["v"] = max(worst["v"], rel_err(v[wi], ov, SCALE["v"]))
        worst["w"] = max(worst["w"], rel_err(w[wi], owv, SCALE["w"]))
        if check_lambda:
            lam, rhs, rs = ow.solution()
            nr = len(lam)
            worst["lam"] = max(worst["lam"], rel_err(con["lam"][wi, :nr], lam, SCALE["lam"]))
    for key in ("p", "R", "v", "w", "geom"):
        assert worst[key] <= tol, f"{key} mismatch {worst[key]:.3e} > {tol}"
    if check_lambda:
        lt = tol if lam_tol is None else lam_tol
        assert worst["lam"] <= lt, f"lambda mismatch {worst['lam']:.3e} > {lt}"
    return worst


def stepwise(scene, nsteps, worlds_idx, batch_kw, oracle_kw, tol=1e-9, lam_tol=1e-9):
    """One step at a time from shared state (the oracle adopts the GPU state before every step):
    compare_step, plus sweep counts and row clamp states bit for bit and the near-tie probe.
    Returns the worst errors."""
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, taps=True, **batch_kw)
    ows = [oracle_world(scene, wi, **oracle_kw)[0] for wi in worlds_idx]
    dt = scene["dt"]
    worst_all = {}
    for s in range(nsteps):
        # shared state: the oracle adopts the GPU state before every step
        p, R, v, w = b.bodies()
        for k, wi in enumerate(worlds_idx):
            ows[k].set_state(p[wi], R[wi], v[wi], w[wi])
        b.step(dt)
        for ow in ows:
            ow.step(dt)
        worst = compare_step(b, ows, worlds_idx, tol=tol, lam_tol=lam_tol)
        st = b.status()
        for k, wi in enumerate(worlds_idx):
            os_ = ows[k].stats()
            assert st["sweeps"][wi] == os_["sweeps"], f"step {s} world {wi}: sweeps {st['sweeps'][wi]} != {os_['sweeps']}"
            lam, rhs, rs = ows[k].solution()
            con = b.contacts()
            con_rs = con["row_state"][wi, :len(rs)]
            assert np.array_equal(con_rs, rs), f"step {s} world {wi}: row clamp states differ"
            # Near-tie probe: the CUDA kernels contract multiply-adds, the oracle does not, so equal clamp
            # states only mean something if no free multiplier sits within rounding distance of a bound.
            # margin = distance of the closest strictly-inside multiplier to its bound (friction rows
            # [-1, 1], normal rows [0, inf)); it must dwarf the CUDA-vs-oracle difference of that world.
            lam = np.asarray(lam); rs = np.asarray(rs)
            # bounded rows: contact blocks, except the first contact block after joints (quirk q2: block c is
            # projected with the bounds of block c - 1, sparse_iterations_utils.cc:169,180,229-235)
            blk = np.arange(len(lam)) // 3
            bounded = (blk > scene["nj"]) if scene["nj"] else np.ones(len(lam), dtype=bool)
            free = (rs == 0) & bounded
            if free.any() and os_["sweeps"] > 0:      # zero sweeps: x is the unprojected initial guess (= rhs)
                row = np.arange(len(lam)) % 3
                dist = np.where(row < 2, 1.0 - np.abs(lam), np.abs(lam))[free]
                diff = float(np.max(np.abs(con["lam"][wi, :len(lam)] - lam)))
                margin = float(dist.min())
                worst_all["clamp_margin"] = min(worst_all.get("clamp_margin", np.inf), margin)
                worst_all["clamp_margin_over_diff"] = min(worst_all.get("clamp_margin_over_diff", np.inf), margin / max(diff, 1e-300))
        assert worst["lam"] <= lam_tol, f"lambda mismatch {worst['lam']:.3e}"
        for k_, v_ in worst.items():
            worst_all[k_] = max(worst_all.get(k_, 0.0), v_)
    b.close()
    if "clamp_margin_over_diff" in worst_all:
        # a free multiplier closer to its bound than ~the rounding difference would make the clamp state a coin toss
        assert worst_all["clamp_margin_over_diff"] > 10.0, f"near-tie: margin {worst_all['clamp_margin']:.3e} is within 10x of the CUDA-vs-oracle difference"
    return worst_all


def stepwise_fp32(scene, nsteps, worlds_idx, batch_kw, oracle_kw, tol=1e-4, sweep_slack=False):
    """`stepwise` for precision = 32 (FP32 constraint records, everything else FP64) against the FP64
    oracle: narrowphase outputs bit-exact, state within `tol` relative, the same sweep counts, no
    status flag.  Returns the worst errors.

    sweep_slack: at converging settings the FP32 records move the residual of a sweep by ~1e-7
    relative, so a sweep count may differ by one, but only where the oracle shows why: its solve
    ended on an exact sweep (final residual < 1e-11; FP32 rounding of 1/(D + cfm) leaves ~1e-8 of
    the previous residual, above the 1e-9 stopping tolerance when that was ~100) and the GPU takes
    one sweep more, or the crossing of the tolerance is a near-tie (the oracle's residual at the
    earlier of the two exit sweeps within 0.1 % of it)."""
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, taps=True, precision=32, **batch_kw)
    ows = [oracle_world(scene, wi, **oracle_kw)[0] for wi in worlds_idx]
    stop = oracle_kw.get("tol", 1e-9)
    worst_all = {}
    for s in range(nsteps):
        p, R, v, w = b.bodies()
        for k, wi in enumerate(worlds_idx):
            ows[k].set_state(p[wi], R[wi], v[wi], w[wi])
        b.step(scene["dt"])
        for ow in ows:
            ow.step(scene["dt"])
        worst = compare_step(b, ows, worlds_idx, tol=tol, check_lambda=False)
        st = b.status()
        assert int(st["status"].max()) == 0
        for k, wi in enumerate(worlds_idx):
            kg, os_ = int(st["sweeps"][wi]), ows[k].stats()
            ko = os_["sweeps"]
            if sweep_slack and abs(kg - ko) == 1:
                if kg == ko + 1 and os_["residual"] < 1e-11:
                    worst_all["exact_sweep_plus_one"] = worst_all.get("exact_sweep_plus_one", 0) + 1
                    continue
                ow2 = oracle_world(scene, wi, **dict(oracle_kw, k_max=min(kg, ko)))[0]
                ow2.set_state(p[wi], R[wi], v[wi], w[wi])
                ow2.step(scene["dt"])
                r = ow2.stats()["residual"]
                assert abs(r / stop - 1.0) < 1e-3, f"step {s} world {wi}: sweeps {kg} != {ko}, oracle residual {r:.6e} at sweep {min(kg, ko)} is no near-tie"
                worst_all["near_tie"] = worst_all.get("near_tie", 0) + 1
                continue
            assert kg == ko, f"step {s} world {wi}: sweeps {kg} != {ko} (oracle residual {os_['residual']:.3e})"
        for key, val in worst.items():
            worst_all[key] = max(worst_all.get(key, 0.0), val)
    b.close()
    assert worst_all["v"] < tol and worst_all["w"] < tol
    return worst_all
