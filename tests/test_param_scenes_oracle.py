"""CPU-side guard of what the scenes of tests/test_gpu_params.py reach, run on the oracle alone: the
box scenes produce every box-box pair code 1-16, the larger minimum constraint distances drop
contacts between box pairs (contact-contact, not only joint-contact), the joint-conflict scenes raise
EGG_ST_JOINT_CONFLICT, and the relaxed stopping tolerances make worlds exit before k_max.  Without
this, an edit of those scenes could turn the GPU tests back into tests of cubes at the reference's
constants without any of them failing."""
import collections

from eggshell_b200 import scenes as S
from tests import test_gpu_params as P
from tests.helpers import oracle_world


def _run(scene, steps, **params):
    """Steps every world of `scene` on the oracle; yields (world, step, oracle world) after each step."""
    for wi in range(scene["W"]):
        ow = oracle_world(scene, wi, **params)[0]
        for s in range(steps):
            ow.step(scene["dt"])
            yield wi, s, ow


def test_box_scenes_reach_every_pair_code():
    """Scenes (a)-(c) at the sizes and step counts of the GPU cases: the pair codes (1-6 face of box 1
    or 2, 7-15 edge-edge, 16 the clipped face with no contact deeper than 1e-9) and the per-pair
    contact counts.  Every code 1-16 must occur."""
    total = collections.Counter()
    for name in ("heap", "crosswise", "rods"):
        build, W, steps = P.BOX_SCENES[name]
        codes, counts = collections.Counter(), collections.Counter()
        for _, _, ow in _run(build(W), steps, solver=1):
            ph = ow.pair_hits()
            codes.update(ph["code"].tolist())
            counts.update(ph["count"].tolist())
        print(f"{name}: pair codes {dict(sorted(codes.items()))}, contacts per pair {dict(sorted(counts.items()))}")
        total.update(codes)
    print("pair-code histogram of scenes (a)-(c):", dict(sorted(total.items())))
    missing = [c for c in range(1, 17) if c not in total]
    assert not missing, f"pair codes never reached: {missing}"


def test_ground_scene_reaches_every_vertex_count():
    """(d): flat boxes touch with 4 vertices, boxes on an edge with 2, on a vertex with 1."""
    build, W, steps = P.BOX_SCENES["ground"]
    seen = set()
    for _, s, ow in _run(build(W), 1, solver=1):
        seen.add(int(ow.stats()["n_contacts"]))
    assert {1, 2, 4} <= seen, seen


def test_dedup_distances_drop_contacts_between_box_pairs():
    """At min_constraint_dist 0.03 and 0.1 every scene of test_dedup_distance_vs_oracle drops contacts
    (stack10, pile64, cairn and the heap have no joints: every drop there is a contact of a box pair
    closer than that to an earlier contact of the same pair); at 0 nothing is dropped."""
    for name in ("stack10", "pile64", "cairn", "chain32", "heap"):
        scene, steps, kw = P._dedup_scene(name)
        for dmin in ((0.0, 0.03) if name == "heap" else (0.0, 0.03, 0.1)):
            dropped = raw = 0
            for _, _, ow in _run(scene, steps, solver=1, min_dist=dmin, **kw):
                st = ow.stats()
                raw += st["n_contacts_raw"]
                dropped += st["n_contacts_raw"] - st["n_contacts"]
            print(f"de-dup {name} min_dist {dmin:g}: {dropped} of {raw} contacts dropped")
            assert (dropped > 0) == (dmin > 0), (name, dmin, dropped)


def test_joint_conflict_scenes_raise_the_flag():
    """rounds at min_constraint_dist 0.25 (hinge joints 0.2 m apart): every world; the coincident chain:
    the even worlds, from init on."""
    flags = [bool(ow.stats()["status"] & 2) for _, _, ow in _run(S.rounds(4), 2, solver=1, k_max=100, min_dist=0.25)]
    assert all(flags)
    sc = P.coincident_chain(6)
    for wi in range(6):
        ow, st0 = oracle_world(sc, wi, solver=1)
        assert bool(st0 & 2) == (wi % 2 == 0), (wi, st0)
        for _ in range(2):
            ow.step(sc["dt"])
            assert bool(ow.stats()["status"] & 2) == (wi % 2 == 0)


def test_relaxed_tol_gives_early_exits():
    """Every (tol, solver) of test_tol_vs_oracle has worlds that stop before k_max."""
    for tol in (1e-6, 1e-3):
        for solver, km in ((1, 500), (2, 6), (3, 40)):
            early = total = 0
            for sc, steps in P.tol_cases(solver):
                for _, _, ow in _run(sc, steps, solver=solver, tol=tol, cfm=0.1, k_max=km):
                    sw = ow.stats()["sweeps"]
                    early += 0 < sw < km
                    total += 1
            print(f"tol {tol:g} solver {solver} k_max {km}: {early} of {total} world-steps exit early")
            assert early > 0, (tol, solver)
