"""Synthetic scene builders for the BASELINE.json configurations (SURVEY.md §8d).

Every scene is a dict of world-major numpy arrays ready for ``Batch.set_bodies/set_joints``:
p,v,w [W,n,3]; R,I [W,n,3,3]; m [W,n]; optional joints i0,i1 [nj], c0,c1 [W,nj,3]; f_ext [W,n,6];
optional box side lengths side [W,n,3] (default 0.3 on every axis); optional Coulomb friction
coefficients mu [W] or a scalar (``Batch.set_friction``); plus ``dt`` and ``solver``.  All bodies are cubes of side 0.3, the only collider the reference has
(/root/reference/eggshell/body.h:90-91).  Randomness is a seeded numpy PCG64 stream per
(config, base seed), so the same arrays feed the GPU batch and the CPU oracle.
"""
import math

import numpy as np

SIDE = 0.3


def quat_to_mat(q):
    """(w,x,y,z) -> rotation matrix, the standard 1-2(y^2+z^2) form."""
    w, x, y, z = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    R = np.empty(q.shape[:-1] + (3, 3))
    R[..., 0, 0] = 1 - 2 * (y * y + z * z)
    R[..., 0, 1] = 2 * (x * y - z * w)
    R[..., 0, 2] = 2 * (x * z + y * w)
    R[..., 1, 0] = 2 * (x * y + z * w)
    R[..., 1, 1] = 1 - 2 * (x * x + z * z)
    R[..., 1, 2] = 2 * (y * z - x * w)
    R[..., 2, 0] = 2 * (x * z - y * w)
    R[..., 2, 1] = 2 * (y * z + x * w)
    R[..., 2, 2] = 1 - 2 * (x * x + y * y)
    return R


def _rot_z(a):
    c, s = np.cos(a), np.sin(a)
    R = np.zeros(np.shape(a) + (3, 3))
    R[..., 0, 0], R[..., 0, 1], R[..., 1, 0], R[..., 1, 1], R[..., 2, 2] = c, -s, s, c, 1.0
    return R


def _rot_x(a):
    c, s = np.cos(a), np.sin(a)
    R = np.zeros(np.shape(a) + (3, 3))
    R[..., 1, 1], R[..., 1, 2], R[..., 2, 1], R[..., 2, 2], R[..., 0, 0] = c, -s, s, c, 1.0
    return R


def _base(W, n):
    return dict(p=np.zeros((W, n, 3)), R=np.tile(np.eye(3), (W, n, 1, 1)), v=np.zeros((W, n, 3)),
                w=np.zeros((W, n, 3)), m=np.ones((W, n)), I=np.tile(np.eye(3) * 0.015, (W, n, 1, 1)),
                n=n, W=W, nj=0)


def chain(W, links=10, anchor=(2.0, 2.0, 1.0), seed=None, anchor_jitter=0.0, v_jitter=0.0, dt=0.001):
    """C1 / C4: Chain(links, anchor) exactly as /root/reference/eggshell/ensembles.cc:668-707.

    Cubes on a body diagonal along +x spaced sqrt(3)*0.3, R = Rz(0.95531661812451) Rx(pi/4),
    joints at the corners (0.15,-0.15,0.15)/(-0.15,0.15,-0.15), link 0's centre anchored to the
    world; m = 1, I = m/12 (0.3^2+0.3^2) = 0.015 (body.cc:19-36)."""
    s = _base(W, links)
    R = _rot_z(np.float64(0.95531661812451)) @ _rot_x(np.float64(math.pi / 4))
    s["R"][:] = R
    a = np.tile(np.asarray(anchor, dtype=np.float64), (W, 1))
    if seed is not None:
        rng = np.random.default_rng(seed)
        a[:, :2] += rng.uniform(-anchor_jitter, anchor_jitter, size=(W, 2))
        s["v"] += rng.uniform(-v_jitter, v_jitter, size=(W, links, 3)) if v_jitter > 0 else 0.0
    s["p"][:, :, 0] = math.sqrt(3.0) * SIDE * np.arange(links)[None, :]
    s["p"] += a[:, None, :]
    nj = links
    i0 = np.concatenate([np.arange(links - 1), [0]]).astype(np.int32)
    i1 = np.concatenate([np.arange(1, links), [-1]]).astype(np.int32)
    c0 = np.tile(np.array([0.15, -0.15, 0.15]), (W, nj, 1))
    c1 = np.tile(np.array([-0.15, 0.15, -0.15]), (W, nj, 1))
    c0[:, -1, :] = 0.0
    c1[:, -1, :] = s["p"][:, 0, :]           # world anchor = initial centre of link 0
    if v_jitter > 0:
        # keep the initial velocity consistent with the anchor: link 0 does not translate
        s["v"][:, 0, :] = 0.0
    s.update(nj=nj, i0=i0, i1=i1, c0=c0, c1=c1, dt=dt, name=f"chain{links}")
    return s


def stack10(W, seed=1000, dt=0.005):
    """C2: 10-box stack on the ground, indexed bottom-up; box k at z = 0.15+0.3k-1e-3(k+1),
    x,y ~ U(+-0.01), yaw ~ U(+-0.05 rad), v = w = 0, m = 1, I = diag(0.015)."""
    n = 10
    s = _base(W, n)
    rng = np.random.default_rng(seed)
    k = np.arange(n)
    s["p"][:, :, 2] = 0.15 + 0.3 * k - 1e-3 * (k + 1)
    s["p"][:, :, :2] = rng.uniform(-0.01, 0.01, size=(W, n, 2))
    s["R"] = _rot_z(rng.uniform(-0.05, 0.05, size=(W, n)))
    s.update(dt=dt, name="stack10")
    return s


def pile64(W, seed=3000, dt=0.005, side=4):
    """C3: side^3 boxes on a lattice of spacing 0.29 (+U(+-0.005)), lowest layer z = 0.14, uniform
    random rotations, v,w ~ U(+-1)^3 (Cairn's limits, ensembles.h:198-199), m = 1, I = 0.1 I3
    (ensembles.cc:719-720)."""
    n = side ** 3
    s = _base(W, n)
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(side), np.arange(side), np.arange(side), indexing="ij"), -1).reshape(-1, 3)
    # index bottom-up: z slowest
    g = g[np.lexsort((g[:, 0], g[:, 1], g[:, 2]))]
    s["p"][:] = 0.29 * g[None, :, :] + rng.uniform(-0.005, 0.005, size=(W, n, 3))
    s["p"][:, :, 2] += 0.14
    s["p"][:, :, :2] -= 0.29 * (side - 1) / 2
    q = rng.normal(size=(W, n, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    s["R"] = quat_to_mat(q)
    s["v"] = rng.uniform(-1, 1, size=(W, n, 3))
    s["w"] = rng.uniform(-1, 1, size=(W, n, 3))
    s["I"] = np.tile(np.eye(3) * 0.1, (W, n, 1, 1))
    s.update(dt=dt, name=f"pile{n}")
    return s


def chain32(W, seed=4000, dt=0.001, anchor_z=0.2122):
    """C4: Chain(32, anchor=(0,0,anchor_z)) lying just above the ground: anchor x,y ~ U(+-0.05),
    v ~ U(+-0.1).  The lowest cube vertices sit 0.2121 below the link centres, so with the default
    anchor_z = 0.2122 the chain lands during the first step and then rests on 30-50 ground contacts
    (186-250 rows, 96 of them the joints' equality rows): the reference's dense Schur + Murty solve
    (lcp.cc:157-336) needs 70-700 pivots per step and succeeds on every step.
    SURVEY.md 8(d) proposed anchor_z = 0.2 (vertices 12 mm INTO the ground): with that start the
    reference's own Murty loop runs into its 1000-pivot cap from step 2 on and MixedConstraintsSolver
    fails, i.e. the reference Panics (ensembles.cc:531-534; reproduced by the oracle, DESIGN.md);
    anchor_z = 0.2 is kept for the PGS golden fixture only."""
    return chain(W, links=32, anchor=(0.0, 0.0, anchor_z), seed=seed, anchor_jitter=0.05, v_jitter=0.1, dt=dt)


def legged20(W, seed=5000, dt=0.005, sigma=0.05):
    """C5: 20-box 'legged' tree: torso (0), 6 legs x (hip, shin, foot) (1..18), head (19), joined by
    19 ball-and-socket joints (the only joint type, joints.h:31); feet 1e-3 into the ground;
    per-world control = constant random torque on the leg links in the f_ext slot
    (ensembles.h:88-89)."""
    n = 20
    s = _base(W, n)
    gap = 0.02
    zf = 0.15 - 1e-3
    zs, zh = zf + SIDE + gap, zf + 2 * (SIDE + gap)
    hips = [(-0.35, -0.35), (0.0, -0.35), (0.35, -0.35), (-0.35, 0.35), (0.0, 0.35), (0.35, 0.35)]
    s["p"][:, 0, :] = (0.0, 0.0, zh)
    i0, i1, c0, c1 = [], [], [], []
    for leg, (hx, hy) in enumerate(hips):
        hip, shin, foot = 1 + 3 * leg, 2 + 3 * leg, 3 + 3 * leg
        s["p"][:, hip, :] = (hx, hy, zh)
        s["p"][:, shin, :] = (hx, hy, zs)
        s["p"][:, foot, :] = (hx, hy, zf)
        # torso-hip joint halfway between the two centres
        mid = np.array([hx / 2, hy / 2, 0.0])
        i0.append(0); i1.append(hip); c0.append(mid); c1.append(mid - np.array([hx, hy, 0.0]))
        h = (SIDE + gap) / 2
        i0.append(hip); i1.append(shin); c0.append((0, 0, -h)); c1.append((0, 0, h))
        i0.append(shin); i1.append(foot); c0.append((0, 0, -h)); c1.append((0, 0, h))
    s["p"][:, 19, :] = (0.0, 0.0, zh + SIDE + gap)
    i0.append(0); i1.append(19); c0.append((0, 0, (SIDE + gap) / 2)); c1.append((0, 0, -(SIDE + gap) / 2))
    nj = len(i0)
    rng = np.random.default_rng(seed)
    f = np.zeros((W, n, 6))
    f[:, :, 2] = -9.8                      # m g with m = 1 (ensembles.cc:218)
    f[:, 1:19, 3:6] = rng.normal(0.0, sigma, size=(W, 18, 3))
    s.update(nj=nj, i0=np.array(i0, dtype=np.int32), i1=np.array(i1, dtype=np.int32),
             c0=np.tile(np.array(c0, dtype=np.float64), (W, 1, 1)), c1=np.tile(np.array(c1, dtype=np.float64), (W, 1, 1)),
             f_ext=f, dt=dt, name="legged20")
    return s


def legged20_motors():
    """The joint motors of legged20 (mpc.Actuators.ball_joint_motors): three per ball joint, 57 for its
    19 joints, acting on the child link and reacting on the parent, with axes in the parent's frame."""
    from .mpc import Actuators
    s = legged20(1)
    return Actuators.ball_joint_motors(s["n"], s["i0"], s["i1"])


def cairn(W, rocks=4, xb=(-0.2, 0.2), yb=(-0.2, 0.2), zb=(1.0, 8.0), seed=7, dt=0.005):
    """Cairn(rocks, bounds) (/root/reference/eggshell/ensembles.cc:709-728) with a seeded stream
    instead of the reference's unseeded std::rand(): random p in the box, uniform random R,
    |v|,|w| components in [-1,1], m = 1, I = 0.1 I3."""
    s = _base(W, rocks)
    rng = np.random.default_rng(seed)
    lo = np.array([min(xb), min(yb), min(zb)])
    hi = np.array([max(xb), max(yb), max(zb)])
    s["p"] = lo + (hi - lo) * rng.uniform(size=(W, rocks, 3))
    q = rng.normal(size=(W, rocks, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    s["R"] = quat_to_mat(q)
    s["v"] = rng.uniform(-1, 1, size=(W, rocks, 3))
    s["w"] = rng.uniform(-1, 1, size=(W, rocks, 3))
    s["I"] = np.tile(np.eye(3) * 0.1, (W, rocks, 1, 1))
    s.update(dt=dt, name=f"cairn{rocks}")
    return s


def hinge(i0, i1, anchor0, anchor1, axis0, axis1, half_span=0.1):
    """A hinge between bodies i0 and i1 as TWO ball-and-socket joints on the hinge axis (the
    reference's only joint type is the 3-row ball joint, joints.h:31; two of them at anchor +-
    half_span * axis leave exactly the rotation about the axis free; the sixth row is redundant and
    is absorbed by cfm).  anchors / axes are given in each body's own frame.  Returns the two
    (i0, i1, c0, c1) tuples to append to a scene's joint lists."""
    a0, a1 = np.asarray(anchor0, float), np.asarray(anchor1, float)
    u0, u1 = np.asarray(axis0, float), np.asarray(axis1, float)
    u0, u1 = u0 / np.linalg.norm(u0), u1 / np.linalg.norm(u1)
    return [(i0, i1, a0 - half_span * u0, a1 - half_span * u1), (i0, i1, a0 + half_span * u0, a1 + half_span * u1)]


def rounds(W, seed=6000, dt=0.005):
    """Mixed colliders (north_star (a): box / sphere / capsule vs ground): 2 boxes, 3 spheres and 3
    capsules per world dropped onto the ground from small heights, two of the spheres overlapping
    (sphere-sphere contact), plus a door: box 1 hinged to box 0 about a vertical axis."""
    n = 8
    s = _base(W, n)
    rng = np.random.default_rng(seed)
    shape = np.array([0, 0, 1, 1, 1, 2, 2, 2], dtype=np.int32)
    dims = np.tile(np.array([[0.3, 0.3, 0.3], [0.3, 0.3, 0.3], [0.12, 0, 0], [0.15, 0, 0], [0.1, 0, 0],
                             [0.08, 0.3, 0], [0.1, 0.2, 0], [0.06, 0.4, 0]]), (W, 1, 1))
    x = np.array([0.0, 0.32, 1.0, 1.2, 2.0, 3.0, 4.0, 5.0])
    s["p"][:, :, 0] = x[None, :] + rng.uniform(-0.01, 0.01, size=(W, n))
    s["p"][:, :, 1] = rng.uniform(-0.01, 0.01, size=(W, n))
    s["p"][:, :, 2] = np.array([0.149, 0.149, 0.118, 0.149, 0.099, 0.2, 0.15, 0.1])[None, :] + rng.uniform(0, 2e-3, size=(W, n))
    q = rng.normal(size=(W, n, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    s["R"] = quat_to_mat(q)
    s["R"][:, :2] = np.eye(3)                       # the two hinged boxes start axis-aligned
    s["p"][:, :2, 1] = 0.0
    s["p"][:, 0, 0] = 0.0; s["p"][:, 1, 0] = 0.32
    s["p"][:, 1, 2] = s["p"][:, 0, 2]               # the hinge anchors coincide exactly
    s["v"] = rng.uniform(-0.2, 0.2, size=(W, n, 3))
    s["v"][:, :2] = 0.0
    s["w"] = rng.uniform(-0.5, 0.5, size=(W, n, 3))
    s["w"][:, :2] = 0.0
    s["I"] = np.tile(np.eye(3) * 0.01, (W, n, 1, 1))
    js = hinge(0, 1, (0.16, 0.0, 0.0), (-0.16, 0.0, 0.0), (0, 0, 1), (0, 0, 1), half_span=0.1)
    s.update(nj=2, i0=np.array([j[0] for j in js], dtype=np.int32), i1=np.array([j[1] for j in js], dtype=np.int32),
             c0=np.tile(np.array([j[2] for j in js]), (W, 1, 1)), c1=np.tile(np.array([j[3] for j in js]), (W, 1, 1)),
             shape=np.tile(shape, (W, 1)), dims=dims, dt=dt, name="rounds")
    return s


def make_batch(scene, **kw):
    """Creates, fills and initialises a ``Batch`` from a scene dict."""
    from .batch import Batch
    b = Batch(scene["W"], scene["n"], scene["nj"], **kw)
    b.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"], side=scene.get("side"))
    if "shape" in scene:
        b.set_shapes(scene["shape"], scene["dims"])
    if scene["nj"]:
        b.set_joints(scene["i0"], scene["i1"], scene["c0"], scene["c1"])
    b.init()
    if "f_ext" in scene:
        b.set_external(scene["f_ext"])
    if "mu" in scene:
        b.set_friction(scene["mu"])
    return b


# Algorithmic HBM bytes per world-step in FP64 (SURVEY.md §8d): read+write the dynamic state
# (18 doubles/body), read the static data (M^-1 10 + f_ext 6 doubles/body), joints (2 int + 6
# double), one cost double out.
def algorithmic_bytes_per_world_step(n, nj):
    return n * (2 * 144 + 128) + 56 * nj + 8
