"""Python host side of the C ABI (include/egg_cuda.h): a batch of W independent ensembles.

Mirrors the reference's ``Ensemble`` interface (/root/reference/eggshell/ensembles.h:25-177):
``init()`` = ``Ensemble::Init``, ``step(dt)`` = ``Ensemble::Step(dt, OPEN_DYNAMICS_ENGINE)``,
``bodies()`` = the ``Body`` accessors, ``contacts()`` = ``Ensemble::constraints()`` taps.  All
compute happens in ``libeggshell_b200.so``; if that library or a CUDA device is missing the
constructor raises — there is no CPU path.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

SOLVER_DENSE_MURTY, SOLVER_PGS, SOLVER_JACOBI, SOLVER_SOR = 0, 1, 2, 3
CFM_AUTO, CFM_ALWAYS, CFM_NEVER = 0, 1, 2
QUIRK_GS_BOUNDS_SHIFT, QUIRK_DENSE_IGNORES_BOUNDS, QUIRKS_REFERENCE = 1, 2, 3
EXPLICIT_EULER, OPEN_DYNAMICS_ENGINE, IMPLICIT_MIDPOINT = 0, 1, 2
ST_LCP_FAILED, ST_JOINT_CONFLICT, ST_BAD_INIT, ST_CONTACT_OVERFLOW, ST_NONFINITE = 1, 2, 4, 8, 16

EXPORTS = [
    "egg_desc_default", "egg_create", "egg_destroy", "egg_set_bodies", "egg_set_shapes", "egg_set_state", "egg_set_joints",
    "egg_set_external", "egg_set_friction", "egg_init", "egg_init_stabilize", "egg_post_stabilize", "egg_step", "egg_step_controlled",
    "egg_set_cost", "egg_step_controlled_cost", "egg_set_actuators", "egg_set_sampler", "egg_sample_controls", "egg_mppi_reduce", "egg_sample_controls_std", "egg_gather_controls", "egg_control_moments", "egg_gather_state", "egg_seed_state", "egg_snapshot", "egg_restore", "egg_update_contacts", "egg_get_static", "egg_get_bodies", "egg_get_contacts", "egg_get_contacts_range", "egg_get_pair_hits", "egg_get_pair_hits_range",
    "egg_get_status", "egg_get_dense_work", "egg_get_debug_counters", "egg_rollout_costs", "egg_set_stream", "egg_sync", "egg_device_bytes",
    "egg_launch_count", "egg_capacity", "egg_get_kernel_config", "egg_set_profiling", "egg_get_kernel_ms", "egg_fp64_peak_tflops", "egg_host_alloc", "egg_host_free", "egg_last_error", "egg_version",
]


class EggDesc(C.Structure):
    _fields_ = [
        ("n_worlds", C.c_int), ("n_bodies", C.c_int), ("n_joints", C.c_int), ("max_contacts", C.c_int),
        ("precision", C.c_int), ("solver", C.c_int), ("k_max", C.c_int),
        ("tol", C.c_double), ("cfm", C.c_double), ("erp", C.c_double), ("gravity", C.c_double * 3),
        ("min_constraint_dist", C.c_double),
        ("quirks", C.c_int), ("cfm_mode", C.c_int), ("device", C.c_int), ("taps", C.c_int),
    ]


class EggCost(C.Structure):
    _fields_ = [
        ("q_run", C.c_void_p), ("l_run", C.c_void_p), ("u_run", C.c_void_p), ("q_term", C.c_void_p),
        ("l_term", C.c_void_p), ("x_ref", C.c_void_p), ("ref_steps", C.c_int),
    ]


class EggSampler(C.Structure):
    _fields_ = [("sigma", C.c_void_p), ("u_lo", C.c_void_p), ("u_hi", C.c_void_p)]


class EggActuators(C.Structure):
    _fields_ = [("m", C.c_int), ("body", C.c_void_p), ("reaction", C.c_void_p), ("frame", C.c_void_p), ("axis", C.c_void_p)]


class EggError(RuntimeError):
    pass


def lib_path():
    return os.path.join(_HERE, "libeggshell_b200.so")


def lib():
    """Loads the CUDA library; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise EggError(f"{path} is missing: run `python -m eggshell_b200.build` (there is no CPU fallback)")
        L = C.CDLL(path)
        L.egg_last_error.restype = C.c_char_p
        L.egg_version.restype = C.c_char_p
        L.egg_device_bytes.restype = C.c_longlong
        L.egg_launch_count.restype = C.c_longlong
        L.egg_host_alloc.restype = C.c_void_p
        L.egg_fp64_peak_tflops.restype = C.c_double
        L.egg_host_alloc.argtypes = [C.c_longlong]
        L.egg_host_free.argtypes = [C.c_void_p]
        L.egg_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.egg_rollout_costs.argtypes = [C.c_void_p, C.c_void_p]
        L.egg_step_controlled.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_int]
        L.egg_set_cost.argtypes = [C.c_void_p, C.c_void_p]
        L.egg_step_controlled_cost.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.egg_gather_state.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.egg_seed_state.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.egg_set_sampler.argtypes = [C.c_void_p, C.c_void_p]
        L.egg_set_actuators.argtypes = [C.c_void_p, C.c_void_p]
        L.egg_sample_controls.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_ulonglong, C.c_ulonglong, C.c_int, C.c_void_p]
        L.egg_mppi_reduce.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        L.egg_sample_controls_std.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_ulonglong, C.c_ulonglong, C.c_int,
                                              C.c_void_p]
        L.egg_gather_controls.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.egg_control_moments.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _LIB = L
    return _LIB


def _chk(rc, what):
    if rc != 0:
        raise EggError(f"{what} failed ({rc}): {lib().egg_last_error().decode()}")


def _d(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        a = np.ascontiguousarray(np.broadcast_to(a, shape))
    return a


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _world_list(worlds, what):
    """A list of world indices as the contiguous int32 array the C ABI takes."""
    w64 = np.asarray(worlds, dtype=np.int64).ravel()
    idx = np.ascontiguousarray(w64, dtype=np.int32)
    if not np.array_equal(idx, w64):
        raise EggError(f"{what}: world index out of the int32 range")
    return idx


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by page-locked host memory (cudaHostAlloc)."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = lib().egg_host_alloc(max(n, 8))
    if not ptr:
        raise EggError("cudaHostAlloc failed")
    buf = (C.c_char * max(n, 8)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr


class Batch:
    """W independent ensembles of n bodies / nj ball joints stepped together on one GPU."""

    def __init__(self, n_worlds, n_bodies, n_joints=0, *, solver=SOLVER_DENSE_MURTY, k_max=500, tol=1e-9,
                 cfm=0.01, erp=0.2, gravity=(0.0, 0.0, -9.8), min_constraint_dist=1e-6, max_contacts=0,
                 quirks=QUIRKS_REFERENCE, cfm_mode=CFM_AUTO, device=0, taps=False, precision=64):
        L = lib()
        d = EggDesc()
        _chk(L.egg_desc_default(C.byref(d), n_worlds, n_bodies, n_joints), "egg_desc_default")
        d.solver, d.k_max, d.tol, d.cfm, d.erp = solver, k_max, tol, cfm, erp
        d.gravity[0], d.gravity[1], d.gravity[2] = gravity
        d.min_constraint_dist, d.max_contacts = min_constraint_dist, max_contacts
        d.quirks, d.cfm_mode, d.device, d.taps = quirks, cfm_mode, device, int(taps)
        d.precision = int(precision)   # 64, or 32 = FP32 constraint records in the PGS stream (opt-in)
        self.h = C.c_void_p()
        _chk(L.egg_create(C.byref(d), C.byref(self.h)), "egg_create")
        self.W, self.n, self.nj = n_worlds, n_bodies, n_joints
        self.desc = d
        self.stream = None   # cudaStream_t handed to set_stream; None = the batch's own stream
        self.cost = None     # mpc.QuadraticCost handed to set_cost
        self.sampler = None  # mpc.MPPI or mpc.CEM handed to set_sampler
        self.actuators = None  # mpc.Actuators handed to set_actuators; None = body wrenches
        self._mu = None        # [W] friction coefficients handed to set_friction; None = BOX friction
        self.max_contacts = None
        self._probe_capacity()

    def _probe_capacity(self):
        self.max_contacts = int(lib().egg_capacity(self.h))
        self.nrec = self.nj + self.max_contacts

    def close(self):
        if self.h:
            lib().egg_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- setup --------------------------------------------------------------------------------
    def set_bodies(self, p, R, v, w, m, I, side=None):
        W, n = self.W, self.n
        p, v, w = _d(p, (W, n, 3)), _d(v, (W, n, 3)), _d(w, (W, n, 3))
        R, I = _d(R, (W, n, 3, 3)), _d(I, (W, n, 3, 3))
        m = _d(m, (W, n))
        s = None if side is None else _d(side, (W, n, 3))
        _chk(lib().egg_set_bodies(self.h, _p(p), _p(R), _p(v), _p(w), _p(m), _p(I), _p(s)), "egg_set_bodies")

    def set_shapes(self, shape, dims):
        """Colliders: 0 box (dims = side lengths), 1 sphere (radius), 2 capsule (radius, axis length)."""
        W, n = self.W, self.n
        shape = np.ascontiguousarray(np.broadcast_to(np.asarray(shape, dtype=np.int32), (W, n)))
        _chk(lib().egg_set_shapes(self.h, _p(shape), _p(_d(dims, (W, n, 3)))), "egg_set_shapes")

    def set_state(self, p=None, R=None, v=None, w=None):
        W, n = self.W, self.n
        a = [None if x is None else _d(x, sh) for x, sh in ((p, (W, n, 3)), (R, (W, n, 3, 3)), (v, (W, n, 3)), (w, (W, n, 3)))]
        _chk(lib().egg_set_state(self.h, *[_p(x) for x in a]), "egg_set_state")

    def set_joints(self, i0, i1, c0, c1):
        W, nj = self.W, self.nj
        i0 = np.ascontiguousarray(np.broadcast_to(np.asarray(i0, dtype=np.int32), (W, nj)))
        i1 = np.ascontiguousarray(np.broadcast_to(np.asarray(i1, dtype=np.int32), (W, nj)))
        c0, c1 = _d(c0, (W, nj, 3)), _d(c1, (W, nj, 3))
        _chk(lib().egg_set_joints(self.h, _p(i0), _p(i1), _p(c0), _p(c1)), "egg_set_joints")

    def set_external(self, f):
        f = _d(f, (self.W, self.n, 6))
        _chk(lib().egg_set_external(self.h, _p(f)), "egg_set_external")

    def set_friction(self, mu):
        """Coulomb-pyramid friction (egg_set_friction, INTEGRATION.md "Friction"): a scalar for every
        world or a [W] array of coefficients, each finite and >= 0; None returns to the reference's BOX
        friction.  PGS solver only.  A refused table leaves the previous one in place."""
        if mu is None:
            _chk(lib().egg_set_friction(self.h, None), "egg_set_friction")
            self._mu = None
            return
        m = _d(mu, (self.W,))
        _chk(lib().egg_set_friction(self.h, _p(m)), "egg_set_friction")
        self._mu = m.copy()

    @property
    def friction(self):
        """A copy of the [W] friction coefficients, or None with BOX friction."""
        return None if self._mu is None else self._mu.copy()

    def init(self):
        _chk(lib().egg_init(self.h), "egg_init")

    def init_stabilize(self, max_steps=100):
        """Ensemble::InitStabilize; returns (relaxation steps taken [W], final squared error [W])."""
        steps = np.zeros(self.W, dtype=np.int32)
        e2 = np.zeros(self.W)
        _chk(lib().egg_init_stabilize(self.h, int(max_steps), _p(steps), _p(e2)), "egg_init_stabilize")
        return steps, e2

    def post_stabilize(self, max_steps=500):
        """Ensemble::PostStabilize; returns (stabilisation steps taken [W], final squared error [W])."""
        steps = np.zeros(self.W, dtype=np.int32)
        e2 = np.zeros(self.W)
        _chk(lib().egg_post_stabilize(self.h, int(max_steps), _p(steps), _p(e2)), "egg_post_stabilize")
        return steps, e2

    def set_stream(self, cuda_stream_ptr):
        _chk(lib().egg_set_stream(self.h, C.c_void_p(cuda_stream_ptr)), "egg_set_stream")
        self.stream = cuda_stream_ptr

    # -- stepping -----------------------------------------------------------------------------
    def step(self, dt, n_steps=1, integrator=OPEN_DYNAMICS_ENGINE):
        _chk(lib().egg_step(self.h, C.c_double(dt), int(integrator), int(n_steps)), "egg_step")

    def step_controlled(self, dt, u_ptr, horizon, integrator=OPEN_DYNAMICS_ENGINE):
        """`horizon` steps; before step t the f_ext slot takes slice t of the device schedule at u_ptr,
        float64 [horizon][W][n][6] (egg_step_controlled), or with an actuator table [horizon][W][m] and
        the slot takes the wrench the table defines."""
        _chk(lib().egg_step_controlled(self.h, C.c_double(dt), int(integrator), C.c_void_p(u_ptr), int(horizon)),
             "egg_step_controlled")

    # -- control space ------------------------------------------------------------------------
    @property
    def control_shape(self):
        """The shape of one world's control row: (n, 6) body wrenches, or (m,) with an actuator table."""
        return (self.n, 6) if self.actuators is None else (self.actuators.m,)

    def set_actuators(self, act):
        """Makes the batch's control row the m values of an mpc.Actuators table for this batch's n
        bodies, or with None the (n, 6) body wrenches again (egg_set_actuators).  Refused while a
        sampler or a cost is set.  Synchronises the batch stream."""
        from .mpc import Actuators
        if act is None:
            _chk(lib().egg_set_actuators(self.h, None), "egg_set_actuators")
        else:
            if not isinstance(act, Actuators) or act.n != self.n:
                raise ValueError(f"set_actuators takes an mpc.Actuators for n = {self.n} bodies, or None")
            a = EggActuators(act.m, _p(act.body), _p(act.reaction), _p(act.frame), _p(act.axis))
            _chk(lib().egg_set_actuators(self.h, C.byref(a)), "egg_set_actuators")
        self.actuators = act

    def _check_control_shape(self, what, obj):
        if obj.control_shape != self.control_shape:
            raise ValueError(f"{what}: the batch's control rows are {self.control_shape}, the {type(obj).__name__}'s "
                             f"{obj.control_shape}")

    def set_cost(self, cost):
        """Configures the cost of step_controlled_cost: an mpc.QuadraticCost for this batch's n bodies
        and control shape, or None to clear it (egg_set_cost).  Synchronises the batch stream."""
        from .mpc import QuadraticCost
        if cost is None:
            _chk(lib().egg_set_cost(self.h, None), "egg_set_cost")
        else:
            if not isinstance(cost, QuadraticCost) or cost.n != self.n:
                raise ValueError(f"set_cost takes an mpc.QuadraticCost for n = {self.n} bodies, or None")
            self._check_control_shape("set_cost", cost)
            c = EggCost(_p(cost.q_run), _p(cost.l_run), _p(cost.u_run), _p(cost.q_term), _p(cost.l_term),
                        _p(cost.x_ref), cost.ref_steps)
            _chk(lib().egg_set_cost(self.h, C.byref(c)), "egg_set_cost")
        self.cost = cost

    def step_controlled_cost(self, dt, u_ptr, horizon, cost_ptr, integrator=OPEN_DYNAMICS_ENGINE):
        """step_controlled that also writes the configured cost J of every world to the device buffer
        at cost_ptr, float64 [W] (egg_step_controlled_cost)."""
        _chk(lib().egg_step_controlled_cost(self.h, C.c_double(dt), int(integrator), C.c_void_p(u_ptr), int(horizon),
                                            C.c_void_p(cost_ptr)), "egg_step_controlled_cost")

    # -- MPPI sampling and weighted reduction --------------------------------------------------
    def set_sampler(self, mppi):
        """Configures the noise scale and control bounds of sample_controls from an mpc.MPPI or mpc.CEM
        (its initial sigma) for this batch's n bodies, or None to clear them (egg_set_sampler).
        Synchronises the batch stream."""
        from .mpc import CEM, MPPI
        if mppi is None:
            _chk(lib().egg_set_sampler(self.h, None), "egg_set_sampler")
        else:
            if not isinstance(mppi, (MPPI, CEM)) or mppi.n != self.n:
                raise ValueError(f"set_sampler takes an mpc.MPPI or mpc.CEM for n = {self.n} bodies, or None")
            self._check_control_shape("set_sampler", mppi)
            s = EggSampler(_p(mppi.sigma), _p(mppi.u_lo), _p(mppi.u_hi))
            _chk(lib().egg_set_sampler(self.h, C.byref(s)), "egg_set_sampler")
        self.sampler = mppi

    def sample_controls(self, u_nom_ptr, horizon, seed, iteration, first, u_ptr):
        """Writes the perturbed schedules float64 [horizon][W][n][6] to the device buffer at u_ptr from
        the nominal schedule [horizon][n][6] at u_nom_ptr (egg_sample_controls).  `first` is the global
        index of local world 0; global world 0 gets no noise."""
        _chk(lib().egg_sample_controls(self.h, C.c_void_p(u_nom_ptr), int(horizon), C.c_ulonglong(int(seed)),
                                       C.c_ulonglong(int(iteration)), int(first), C.c_void_p(u_ptr)), "egg_sample_controls")

    def mppi_reduce(self, u_ptr, horizon, cost_ptr, baseline_ptr, lam, out_ptr):
        """out (device, float64 [horizon n 6 + 2]) = sum_w omega_w u[t][w], sum omega, sum omega^2 with
        omega_w = exp(-(cost[w] - baseline) / lam), 0 for a non-finite cost (egg_mppi_reduce).
        baseline_ptr is a device scalar."""
        _chk(lib().egg_mppi_reduce(self.h, C.c_void_p(u_ptr), int(horizon), C.c_void_p(cost_ptr), C.c_void_p(baseline_ptr),
                                   C.c_double(lam), C.c_void_p(out_ptr)), "egg_mppi_reduce")

    # -- CEM sampling and elite refit ----------------------------------------------------------
    def sample_controls_std(self, mean_ptr, std_ptr, horizon, seed, iteration, first, u_ptr):
        """sample_controls with a per-step noise scale: u[t][w] = clamp(mean[t] + std[t] eps) from the
        device arrays float64 [horizon][n][6] at mean_ptr and std_ptr, with the eps of sample_controls
        (egg_sample_controls_std).  The bounds are the sampler's; its sigma is not used."""
        _chk(lib().egg_sample_controls_std(self.h, C.c_void_p(mean_ptr), C.c_void_p(std_ptr), int(horizon), C.c_ulonglong(int(seed)),
                                           C.c_ulonglong(int(iteration)), int(first), C.c_void_p(u_ptr)), "egg_sample_controls_std")

    def gather_controls(self, u_ptr, horizon, worlds, out_ptr):
        """Copies the schedules of the listed local worlds out of the device buffer at u_ptr, float64
        [horizon][W][n][6], to the device buffer at out_ptr, [len(worlds)][horizon][n][6]
        (egg_gather_controls)."""
        idx = _world_list(worlds, "gather_controls")
        _chk(lib().egg_gather_controls(self.h, C.c_void_p(u_ptr), int(horizon), _p(idx), int(idx.size), C.c_void_p(out_ptr)),
             "egg_gather_controls")

    def control_moments(self, rows_ptr, k, horizon, out_ptr):
        """out (device, float64 [2][horizon][n][6]) = the mean and the population standard deviation of
        the k rows [k][horizon][n][6] at rows_ptr, summed in row order (egg_control_moments)."""
        _chk(lib().egg_control_moments(self.h, C.c_void_p(rows_ptr), int(k), int(horizon), C.c_void_p(out_ptr)),
             "egg_control_moments")

    # -- device-side state exchange (MPC) ------------------------------------------------------
    def gather_state(self, worlds, out_ptr):
        """Writes the state of the listed worlds to the device buffer at out_ptr, float64
        [len(worlds)][n][18] = (p, R row-major, v, w) per body (egg_gather_state)."""
        idx = _world_list(worlds, "gather_state")
        _chk(lib().egg_gather_state(self.h, _p(idx), int(idx.size), C.c_void_p(out_ptr)), "egg_gather_state")

    def seed_state(self, in_ptr, k, first=0):
        """World w takes row (first + w) % k of the device buffer at in_ptr, float64 [k][n][18]
        (egg_seed_state).  Call snapshot() to make the seeded state the next horizon's start."""
        _chk(lib().egg_seed_state(self.h, C.c_void_p(in_ptr), int(k), int(first)), "egg_seed_state")

    def update_contacts(self):
        _chk(lib().egg_update_contacts(self.h), "egg_update_contacts")

    def static(self):
        W, n = self.W, self.n
        ml, ma, f = np.empty((W, n)), np.empty((W, n, 3, 3)), np.empty((W, n, 6))
        _chk(lib().egg_get_static(self.h, _p(ml), _p(ma), _p(f)), "egg_get_static")
        return ml, ma, f

    def snapshot(self):
        _chk(lib().egg_snapshot(self.h), "egg_snapshot")

    def restore(self):
        _chk(lib().egg_restore(self.h), "egg_restore")

    def sync(self):
        _chk(lib().egg_sync(self.h), "egg_sync")

    # -- readback -----------------------------------------------------------------------------
    def bodies(self, out=None):
        W, n = self.W, self.n
        if out is None:
            out = (np.empty((W, n, 3)), np.empty((W, n, 3, 3)), np.empty((W, n, 3)), np.empty((W, n, 3)))
        p, R, v, w = out
        _chk(lib().egg_get_bodies(self.h, _p(p), _p(R), _p(v), _p(w)), "egg_get_bodies")
        return p, R, v, w

    def contacts(self, first=0, n_worlds=None):
        """Contact taps of the last step; `first` / `n_worlds` select a world range (default: all)."""
        W = self.W - first if n_worlds is None else n_worlds
        mc, nr = self.max_contacts, self.nrec
        count = np.zeros(W, dtype=np.int32)
        i0, i1, code = (np.zeros((W, mc), dtype=np.int32) for _ in range(3))
        pos, nrm, depth = np.zeros((W, mc, 3)), np.zeros((W, mc, 3)), np.zeros((W, mc))
        lam = np.zeros((W, 3 * nr))
        rs = np.zeros((W, 3 * nr), dtype=np.int32)
        _chk(lib().egg_get_contacts_range(self.h, int(first), int(W), _p(count), _p(i0), _p(i1), _p(pos), _p(nrm), _p(depth),
                                          _p(code), _p(lam), _p(rs)), "egg_get_contacts_range")
        return dict(count=count, i0=i0, i1=i1, pos=pos, nrm=nrm, depth=depth, code=code, lam=lam, row_state=rs)

    def pair_hits(self):
        W, P = self.W, max(1, self.n * (self.n - 1) // 2)
        nh = np.zeros(W, dtype=np.int32)
        a = [np.zeros((W, P), dtype=np.int32) for _ in range(4)]
        _chk(lib().egg_get_pair_hits(self.h, _p(nh), *[_p(x) for x in a], P), "egg_get_pair_hits")
        return dict(n=nh, i=a[0], j=a[1], code=a[2], count=a[3])

    def status(self):
        W = self.W
        st = np.zeros(W, dtype=np.int32)
        stats = np.zeros((W, 8), dtype=np.int32)
        res = np.zeros(W)
        _chk(lib().egg_get_status(self.h, _p(st), _p(stats), _p(res)), "egg_get_status")
        return dict(status=st, n_contacts_raw=stats[:, 0], n_contacts=stats[:, 1], n_rows=stats[:, 2],
                    n_pair_hits=stats[:, 3], sweeps=stats[:, 4], pivots=stats[:, 5], cfm_applied=stats[:, 6],
                    residual=res)

    def dense_work(self):
        """FP64 operations of the reference algorithm on each world's last dense solve [W]."""
        out = np.zeros(self.W)
        _chk(lib().egg_get_dense_work(self.h, _p(out)), "egg_get_dense_work")
        return out

    def debug_counters(self, reset=True):
        out = np.zeros(32, dtype=np.uint64)
        _chk(lib().egg_get_debug_counters(self.h, _p(out), int(reset)), "egg_get_debug_counters")
        return out

    def rollout_costs(self, device_ptr):
        _chk(lib().egg_rollout_costs(self.h, C.c_void_p(device_ptr)), "egg_rollout_costs")

    def kernel_config(self):
        """The kernel instances this batch runs (egg_get_kernel_config): lanes per world, worlds per
        warp, M^-1 layout (-1 until the first step), record format (-1 until the first step for PGS),
        run cap, record precision, narrowphase and record-assembly threads per world."""
        out = (C.c_int * 8)()
        _chk(lib().egg_get_kernel_config(self.h, out), "egg_get_kernel_config")
        keys = ("lpw", "worlds_per_warp", "iso", "rec_format", "run_cap", "precision", "collide_threads", "records_threads")
        return dict(zip(keys, (int(x) for x in out)))

    def set_profiling(self, on=True):
        _chk(lib().egg_set_profiling(self.h, int(on)), "egg_set_profiling")

    def kernel_ms(self):
        """(narrowphase, assembly, solve+integrate) device milliseconds and the steps they cover."""
        out = np.zeros(4)
        _chk(lib().egg_get_kernel_ms(self.h, _p(out)), "egg_get_kernel_ms")
        return out

    @property
    def device_bytes(self):
        return lib().egg_device_bytes(self.h)

    @property
    def launch_count(self):
        return lib().egg_launch_count(self.h)


def fp64_peak_tflops(device=0):
    v = lib().egg_fp64_peak_tflops(int(device))
    if v < 0:
        raise EggError(f"egg_fp64_peak_tflops failed ({v}): {lib().egg_last_error().decode()}")
    return v
