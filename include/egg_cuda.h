/* egg_cuda.h — C ABI of the B200 batched rigid-body step (libeggshell_b200.so).
 *
 * The reference (teenylasers/eggshell) has no plugin/FFI: its boundary is the C++ link-time
 * surface `Ensemble::{Init,Step}` (/root/reference/eggshell/ensembles.h:25-177) driven by
 * `SimulationInitialization()/SimulationStep()` (/root/reference/eggshell/model.h:8-13).  Each
 * entry point below names the reference interface it replaces.  The source-compatible C++ mirror
 * of those headers (include/eggshell/) forwards to this ABI; see INTEGRATION.md.
 *
 * Conventions: every pointer is a HOST pointer unless the name ends in _d (device).  Host arrays
 * are array-of-structs in world-major order: [world][body][k] or [world][joint][k]; matrices are
 * 3x3 row-major.  All functions return 0 on success or a negative egg_error; nothing aborts the
 * process and no exception crosses the boundary (the reference's Panic()/_exit(1),
 * /root/reference/toolkit/error.cc:44-49, becomes a per-world status word).  One host thread
 * drives one batch; calls on one batch are not thread-safe (same contract as the reference's
 * single GUI thread, /root/reference/eggshell/eggshell_view.cc:540-554).
 */
#ifndef EGG_CUDA_H_
#define EGG_CUDA_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct egg_batch egg_batch; /* opaque: owns all device memory of W independent worlds */

enum egg_error {
  EGG_OK = 0,
  EGG_ERR_ARG = -1,       /* bad argument / descriptor */
  EGG_ERR_CUDA = -2,      /* a CUDA runtime call failed; see egg_last_error() */
  EGG_ERR_NO_DEVICE = -3, /* no CUDA device: there is NO CPU fallback */
  EGG_ERR_STATE = -4,     /* call order violated (e.g. egg_step before egg_init) */
  EGG_ERR_UNSUPPORTED = -5
};

/* ensembles.h:45-49 enum Integrator.  Only OPEN_DYNAMICS_ENGINE works with contacts in the
 * reference (ensembles.cc:398-405); the others return EGG_ERR_UNSUPPORTED. */
enum egg_integrator { EGG_EXPLICIT_EULER = 0, EGG_OPEN_DYNAMICS_ENGINE = 1, EGG_IMPLICIT_MIDPOINT = 2 };

/* Which solver ComputeVDot uses.  0 is what the reference ships (ensembles.cc:21,531);
 * 1..3 are sparse_iterations.h:26-34 wired into the same slot. */
enum egg_solver { EGG_SOLVER_DENSE_MURTY = 0, EGG_SOLVER_PGS = 1, EGG_SOLVER_JACOBI = 2, EGG_SOLVER_SOR = 3 };

/* Constraint-force-mixing policy on the dense path (ensembles.cc:514-521).  AUTO reproduces the
 * reference's "condition number >= 1e7 => add cfm" decision. */
enum egg_cfm_mode { EGG_CFM_AUTO = 0, EGG_CFM_ALWAYS = 1, EGG_CFM_NEVER = 2 };

/* Reference quirks kept behind flags (SURVEY.md §8 q1,q2); EGG_QUIRKS_REFERENCE = both on. */
enum egg_quirk {
  EGG_QUIRK_GS_BOUNDS_SHIFT = 1,      /* sparse_iterations_utils.cc:169,180,229-235 */
  EGG_QUIRK_DENSE_IGNORES_BOUNDS = 2, /* lcp.cc:298 -> :141-147 */
  /* Not a reference quirk: keep (R I_b R^T)^-1 exactly as computed (ensembles.cc:210).  By default
   * egg_init snaps a numerically isotropic inverse inertia (|dev| <= 1e-13 relative; every body of
   * the reference's own scenes) to c^-1 I3, which lets the PGS kernel keep 2 doubles per body. */
  EGG_OPT_EXACT_INERTIA = 4,
  /* Not a reference quirk: run the 15-axis SAT on every body pair.  By default pairs whose bounding
   * spheres are clearly apart are culled first (conservative: the colliding-pair list is unchanged). */
  EGG_OPT_NO_BROADPHASE_CULL = 8,
  /* Not a reference quirk: the run format of the PGS record stream (egg_pgs_runs.cu): a lane carries
   * the consecutive contacts of one manifold through a stage, records shrink to 80 B per block +
   * 64 B per run.  Same sweep in the same row order; measured faster only for stack-like scenes
   * (DESIGN.md section 4), so it is opt-in.  Isotropic bodies, FP64 records only, and no friction
   * table (egg_set_friction): else ignored, decided at every step. */
  EGG_OPT_PGS_RUNS = 16
};
#define EGG_QUIRKS_REFERENCE 3

/* Per-world status bits (egg_get_status). */
enum egg_status {
  EGG_ST_OK = 0,
  EGG_ST_LCP_FAILED = 1,        /* ensembles.cc:531-534 would Panic */
  EGG_ST_JOINT_CONFLICT = 2,    /* ensembles.cc:280-285 would Panic */
  EGG_ST_BAD_INIT = 4,          /* ensembles.cc:27 CHECK_MSG would fail */
  EGG_ST_CONTACT_OVERFLOW = 8,  /* more contacts than max_contacts; the tail was dropped */
  EGG_ST_NONFINITE = 16,        /* NaN/Inf reached the state */
  EGG_ST_DENSE_OVERFLOW = 32,   /* more rows than the dense path is provisioned for; lambda = 0 */
  EGG_ST_INTERNAL = 64          /* a staged constraint record failed its range check inside the solve kernel (never expected;
                                   the block is skipped instead of dereferencing a bad index) */
};

/* Compile-time constants of the reference gathered into one POD (SURVEY.md §5 "Config"):
 * constants.h:5-12, ensembles.cc:14-21, ensembles.h:165-166, sparse_iterations.cc:15-19. */
typedef struct egg_desc {
  int n_worlds;     /* W independent ensembles */
  int n_bodies;     /* bodies per world (Ensemble::n_, ensembles.h:75) */
  int n_joints;     /* ball-and-socket joints per world (ensembles.h:81) */
  int max_contacts; /* per-world contact capacity after de-duplication; 0 = automatic */
  int precision;    /* 64 (FP64, reference arithmetic).  32 (opt-in, PGS solver only): the constraint records of
                       the solve are stored in FP32 (40 % fewer bytes in an HBM-bound kernel); narrowphase,
                       assembly arithmetic, multipliers, accumulators and the integrator stay FP64, so
                       the discrete outputs of the narrowphase are unchanged and the state agrees with
                       the FP64 path to ~1e-6 relative per step (tested at 1e-4) */
  int solver;       /* egg_solver */
  int k_max;        /* kNumIterations = 500 */
  double tol;       /* kAllowNumericalError = 1e-9 */
  double cfm;       /* kCfmCoeff = 0.01 */
  double erp;       /* error_reduction_param = 0.2 */
  double gravity[3];            /* kGravity = (0,0,-9.8) */
  double min_constraint_dist;   /* kMinConstraintDistance = 1e-6 */
  int quirks;       /* egg_quirk bitmask; EGG_QUIRKS_REFERENCE for parity */
  int cfm_mode;     /* egg_cfm_mode */
  int device;       /* CUDA device ordinal */
  int taps;         /* 1 = keep per-pair parity taps (egg_get_pair_hits); costs memory */
} egg_desc;

/* Fills *d with the reference defaults for the given shape. */
int egg_desc_default(egg_desc* d, int n_worlds, int n_bodies, int n_joints);

/* Ensemble construction (ensembles.h:25-29 + the Chain/Cairn ctors, ensembles.cc:668-728). */
int egg_create(const egg_desc* d, egg_batch** out);
void egg_destroy(egg_batch* b);

/* Body state: Body::{p_,R_,v_,w_,m_,I_,side_lengths_} (body.h:79-91).  side may be NULL
 * (0.3,0.3,0.3 as body.h:91). */
int egg_set_bodies(egg_batch* b, const double* p, const double* R, const double* v, const double* w,
                   const double* m, const double* I_body, const double* side);
/* Colliders other than the reference's box (BASELINE.json north_star (a); the reference only draws
 * spheres and capsules, model.h:16-25, so the contact rules are this project's, defined by
 * oracle/orc_collision.h: parity unpinned).  shape[W][n]: 0 box (dims = side lengths, the default),
 * 1 sphere (dims[0] = radius), 2 capsule (dims[0] = radius, dims[1] = length of the axis segment along
 * the body's z axis); dims[W][n][3].  Ground contacts: the lowest point of every (end) sphere below
 * z = 0; pairs: box-box (the reference's SAT) and sphere-sphere (one contact, code 17); other
 * collider pairs generate no contacts.  Call after egg_set_bodies; mass and inertia stay the caller's. */
int egg_set_shapes(egg_batch* b, const int* shape, const double* dims);

/* Dynamic state only (SetP/SetR/SetV/SetW_GlobalFrame, body.h:64-71).  The host-to-device copies
 * are asynchronous on the batch stream: when the arrays live in pinned memory (egg_host_alloc) the
 * call returns before they have been read, so keep them unchanged until the next synchronising
 * call (egg_sync, egg_get_*).  Pageable arrays are staged by the runtime before the call returns. */
int egg_set_state(egg_batch* b, const double* p, const double* R, const double* v, const double* w);
/* BallAndSocketJoint(b0,i0,c0,b1,i1,c1) / (b0,i0,c0,c1_world) (joints.h:34-42); i1 = -1 anchors
 * body i0 to the world point c1. */
int egg_set_joints(egg_batch* b, const int* i0, const int* i1, const double* c0, const double* c1);
/* Overrides Ensemble::external_force_torque_ (ensembles.h:88-89) after egg_init; 6 per body. */
int egg_set_external(egg_batch* b, const double* f_ext);

/* Coulomb-pyramid friction with one coefficient per world (INTEGRATION.md, "Friction").  mu is a HOST
 * [n_worlds] array, each entry finite and >= 0; it is copied to device memory owned by the batch
 * (counted by egg_device_bytes).  With a table, the PGS solve bounds the two tangent rows of a block
 * projected as a contact by [-b, b], b = mu[w] max(x_n, 0), x_n the block's normal multiplier before
 * its update, instead of the reference's BOX bounds [-1, 1]; a tangent row is "at its bound" in the
 * residual and in the row_state taps when that projection clamped it.  mu == NULL returns to BOX
 * friction, bit for bit, and releases the memory.  EGG_ERR_ARG for a NaN, infinite or negative entry
 * (the previous table is kept); EGG_ERR_UNSUPPORTED unless the solver is EGG_SOLVER_PGS (the dense
 * path, Jacobi and SOR keep BOX friction).  While a table is set the run format (EGG_OPT_PGS_RUNS) is
 * not used.  Valid before or after egg_init.  Synchronises the batch stream. */
int egg_set_friction(egg_batch* b, const double* mu);

/* Ensemble::Init (ensembles.cc:24-29): M^-1 blocks, f_ext, initial-condition check and
 * CheckAndCorrectEnsembleState (a joint-joint conflict sets EGG_ST_JOINT_CONFLICT here, where the
 * reference Panics).  Body state changed afterwards reaches the device only through
 * egg_set_state / egg_set_bodies. */
int egg_init(egg_batch* b);

/* Ensemble::InitStabilize (ensembles.cc:602-622): refresh contacts, and while a world's squared
 * position error exceeds 1e-9 (and fewer than max_steps relaxations were taken, 100 in the
 * reference) apply StepPositionRelaxation(dt = 0.5, step_scale = 0.2); finally
 * CheckAndCorrectEnsembleState.  steps_out[W] / err_sq_out[W] may be NULL.  Synchronous. */
int egg_init_stabilize(egg_batch* b, int max_steps, int* steps_out, double* err_sq_out);

/* Ensemble::PostStabilize(max_steps) (ensembles.cc:624-645, max_steps = 500 in ensembles.h:59):
 * while a world's squared position error exceeds 1e-9 apply StepPostStabilization(dt = 0.1,
 * step_scale = 0.2) (ensembles.cc:652-657): positions AND velocities move by the relaxation
 * -0.2 J^T (J J^T)^-1 err.  As in the reference the contact list is not refreshed inside the loop
 * (a contact's error is its stored depth).  steps_out[W] / err_sq_out[W] may be NULL.  Synchronous. */
int egg_post_stabilize(egg_batch* b, int max_steps, int* steps_out, double* err_sq_out);

/* n_steps x Ensemble::Step(dt, integrator) (ensembles.cc:390-427) on every world; asynchronous on
 * the batch stream. */
int egg_step(egg_batch* b, double dt, int integrator, int n_steps);

/* Receding-horizon MPC (INTEGRATION.md).  The three calls below take DEVICE buffers on the batch's
 * device (cudaPointerGetAttributes must report device or managed memory there, else EGG_ERR_ARG);
 * their lengths cannot be checked through a raw pointer and are the caller's responsibility.  They
 * are asynchronous on the batch stream: keep the buffers alive and unchanged until the next
 * synchronising call.  Before egg_init they return EGG_ERR_STATE. */

/* horizon x Ensemble::Step(dt, integrator) with a per-step control schedule: before step t the f_ext
 * slot of every world is replaced by u_d[t], exactly what egg_set_external(u[t]) before
 * egg_step(b, dt, integrator, 1) does.  u_d is [horizon][W][n_bodies][6], time-major, so every slice
 * has the layout of egg_set_external.  After the call the slot holds u_d[horizon-1].  horizon >= 1.
 * With an actuator table (egg_set_actuators) u_d is [horizon][W][m] and the slot takes the wrench the
 * table defines from u_d[t] and the state before step t. */
int egg_step_controlled(egg_batch* b, double dt, int integrator, const double* u_d, int horizon);

/* Actuators: a control space of m actuator values per world in place of the n_bodies x 6 body wrenches,
 * shared by all worlds of the batch (INTEGRATION.md, "Actuators").  Actuator a applies the torque
 * +tau_a to body[a] (in [0, n_bodies)) and -tau_a to reaction[a] (in [-1, n_bodies), != body[a]; -1 =
 * none).  Its axis axis[a][3] (finite, not all zero, used as given: its length is the gear ratio) is
 * given in the rotation of body frame[a] (-1, body[a] or reaction[a]; -1 = the world frame).  With x_t
 * the state before step t (the row the running cost reads) and u_a the actuator value of step t:
 *   k_a = axis[a]                         if frame[a] = -1
 *       = R k, (R k)_i = (R_i0 k_0 + R_i1 k_1) + R_i2 k_2,   R = R of body frame[a] in x_t
 *   tau_a = u_a k_a                       (component-wise)
 *   f_ext[b] = (m_b g_x, m_b g_y, m_b g_z, 0, 0, 0), then for a = 0 .. m-1 in order:
 *              torque += tau_a if body[a] = b;  torque -= tau_a if reaction[a] = b
 * Every product and sum is rounded on its own (no fused multiply-add), so a float64 transcription in
 * the same order (mpc.Actuators.wrench) has the same bits.  The base wrench is the force part of the
 * slot egg_init writes (m g from the mass and egg_desc.gravity, the same product); the gyroscopic
 * torque egg_init freezes into the slot is NOT included.  It is zero for worlds at rest at egg_init.
 * The wrench is held over step t (zero-order hold, like f_ext in the reference); after a controlled
 * call the slot holds the wrench of the last step.  An actuator table adds no forces: body-force
 * controls stay available in the default control space. */
typedef struct egg_actuators {
  int m;               /* number of actuators, >= 1 */
  const int* body;     /* [m] (every array is a HOST array) */
  const int* reaction; /* [m] */
  const int* frame;    /* [m] */
  const double* axis;  /* [m][3] */
} egg_actuators;

/* Sets the batch's actuator table: copies it to device memory owned by the batch (counted by
 * egg_device_bytes), with a per-body list of the actuators that touch each body, in actuator order.
 * a == NULL returns to body wrenches and releases that memory.  From then on the control row per world
 * of every call below is the m actuator values: u_d [H][W][m] (egg_step_controlled,
 * egg_step_controlled_cost, egg_sample_controls, egg_sample_controls_std, egg_mppi_reduce,
 * egg_gather_controls), u_nom_d / mean_d / std_d [H][m], egg_sampler sigma, u_lo, u_hi [m], egg_cost
 * u_run [m], egg_mppi_reduce out_d [H m + 2], egg_gather_controls out_d [k][H][m] and
 * egg_control_moments rows_d [k][H][m], out_d [2][H][m]; their checks apply to that width.  A
 * malformed table returns EGG_ERR_ARG and keeps the previous one.  EGG_ERR_STATE while a sampler or a
 * cost is set: their arrays have the width of the current control space, clear them first.  Valid
 * before or after egg_init.  Synchronises the batch stream. */
int egg_set_actuators(egg_batch* b, const egg_actuators* a);

/* out_d[k][n_bodies][18] = (p(3), R(9, row-major), v(3), w(3)) of worlds[0..k), element for element
 * what egg_get_bodies returns for those worlds.  worlds is a HOST int array, each entry in [0, W),
 * duplicates allowed; 1 <= k <= W. */
int egg_gather_state(egg_batch* b, const int* worlds, int k, double* out_d);

/* World w takes the state in_d[(first + w) mod k] (the [k][n_bodies][18] layout of egg_gather_state);
 * 1 <= k <= W, first >= 0.  first is the global index of local world 0 of a sharded sweep, so a
 * world's seed does not depend on the sharding.  Only the live state is written: call egg_snapshot
 * to make it the start of the next horizon.  The rollout cost keeps its egg_init reference pose. */
int egg_seed_state(egg_batch* b, const double* in_d, int k, int first);

/* A quadratic running + terminal cost over a controlled horizon, shared by all worlds.  A body's
 * state row is x = (p(3), R(9, row-major), v(3), w(3)) (the egg_gather_state row), its control
 * u = (f(3), tau(3)) (the egg_set_external row).  With x_t the state before step t, x_H the state
 * after the last step and d_t = x_t - x_ref[t] (x_ref[t] = x_ref[0] when ref_steps = 1):
 *   J = sum_{t<H} sum_b [ sum_c q_run[b][c] d_t[b][c]^2 + l_run[b][c] d_t[b][c] + sum_j u_run[b][j] u_t[b][j]^2 ]
 *     +           sum_b   sum_c q_term[b][c] d_H[b][c]^2 + l_term[b][c] d_H[b][c]
 * The linear terms express progress (l_term[0][0] = -1: reward body 0 for moving along +x).
 * Non-finite states or controls propagate into J as computed. */
typedef struct egg_cost {
  const double* q_run;  /* [n_bodies][18]; NULL = all zero (every array is a HOST array) */
  const double* l_run;  /* [n_bodies][18] */
  const double* u_run;  /* [n_bodies][6]; [m] with an actuator table (egg_set_actuators) */
  const double* q_term; /* [n_bodies][18] */
  const double* l_term; /* [n_bodies][18] */
  const double* x_ref;  /* [ref_steps][n_bodies][18]; NULL = zeros (ref_steps is then ignored) */
  int ref_steps;        /* 1 (a constant reference) or >= horizon + 1 of every later rollout */
} egg_cost;

/* Copies the cost into device memory owned by the batch (counted by egg_device_bytes); c == NULL
 * clears it and releases that memory.  Non-finite weights or reference values, or ref_steps < 1 with
 * a reference, return EGG_ERR_ARG and leave the previous cost in place.  Valid before or after
 * egg_init.  Synchronises the batch stream. */
int egg_set_cost(egg_batch* b, const egg_cost* c);

/* egg_step_controlled, bit for bit the same state and f_ext slot, that also writes J of every world
 * (the cost of egg_set_cost) to the DEVICE buffer cost_d[W].  cost_d is overwritten, not added to.
 * The sum runs in an order that depends only on n_bodies and the step, so a world's J has the same
 * bits in any batch.  EGG_ERR_STATE without a cost or before egg_init; EGG_ERR_ARG for the arguments
 * egg_step_controlled refuses, a cost_d that is not device memory of the batch's device, or
 * 1 < ref_steps < horizon + 1.  Every check runs before the first launch; asynchronous on the
 * batch stream. */
int egg_step_controlled_cost(egg_batch* b, double dt, int integrator, const double* u_d, int horizon, double* cost_d);

/* MPPI (model predictive path integral, INTEGRATION.md): the two data-heavy steps of a sampling
 * planner, sampling W perturbed copies of a nominal schedule and their cost-weighted sum.
 * Per-body noise scale and control bounds, shared by all worlds and steps: */
typedef struct egg_sampler {
  const double* sigma; /* [n_bodies][6] standard deviation of the noise, finite and >= 0 (HOST array); [m] with an actuator table */
  const double* u_lo;  /* [n_bodies][6] lower bound of every sampled control; NULL = unbounded */
  const double* u_hi;  /* [n_bodies][6] upper bound; NULL = unbounded.  +-inf allowed, NaN not */
} egg_sampler;

/* Copies the sampler into device memory owned by the batch (counted by egg_device_bytes); s == NULL
 * clears it and releases that memory.  A non-finite or negative sigma, a NaN bound or u_lo > u_hi
 * returns EGG_ERR_ARG and leaves the previous sampler in place.  Valid before or after egg_init.
 * Synchronises the batch stream. */
int egg_set_sampler(egg_batch* b, const egg_sampler* s);

/* u_d[t][w][b][j] = clamp(u_nom_d[t][b][j] + sigma[b][j] eps, u_lo[b][j], u_hi[b][j]) for t < horizon
 * and every local world w; u_nom_d is [horizon][n_bodies][6], u_d [horizon][W][n_bodies][6] (the
 * schedule of egg_step_controlled).  eps is a standard normal from Philox4x32-10 with key
 * (seed_lo, seed_hi) and counter (q, g, iteration_lo, iteration_hi), g = first + w the global world
 * index and q = (t n_bodies + b) 3 + p for the component pair (2p, 2p + 1) (in general q = t ceil(c / 2)
 * + p for the elements (2p, 2p + 1) of a control row of width c; with an actuator table c = m, and for
 * odd m the last pair discards its second normal): the four output words
 * make two uniforms u = ((lo | hi << 32) >> 11) 2^-53 + 2^-54 (words 0, 1 and words 2, 3), and
 * Box-Muller gives eps_2p = r cos(2 pi u2), eps_2p+1 = r sin(2 pi u2), r = sqrt(-2 ln u1).  The
 * samples depend on the global index only, not on the sharding.  Global world 0 takes no noise: it
 * runs clamp(u_nom).  EGG_ERR_STATE without a sampler or before egg_init; EGG_ERR_ARG for
 * horizon < 1, first < 0, or a pointer that is not device memory of the batch's device.
 * Asynchronous on the batch stream; one launch. */
int egg_sample_controls(egg_batch* b, const double* u_nom_d, int horizon, unsigned long long seed,
                        unsigned long long iteration, int first, double* u_d);

/* The cost-weighted sum of the schedules u_d [horizon][W][n_bodies][6].  World w gets the weight
 * omega_w = exp(-(cost_d[w] - *baseline_d) / lambda); omega_w = 0 for a non-finite cost_d[w], and every
 * weight is 0 when *baseline_d (a DEVICE scalar) is not finite.  out_d [horizon n_bodies 6 + 2]
 * receives sum_w omega_w u_d[t][w] as [horizon][n_bodies][6], then sum omega, then sum omega^2.
 * Deterministic, without atomics: each fixed chunk of worlds is summed in index order into a scratch
 * buffer the batch owns (counted by egg_device_bytes), then the chunk sums are added in chunk order,
 * so the bits depend only on W, n_bodies, horizon and the inputs.  EGG_ERR_ARG for lambda <= 0 or
 * not finite, horizon < 1, or a pointer that is not device memory of the batch's device;
 * EGG_ERR_STATE before egg_init.  Asynchronous on the batch stream; two launches. */
int egg_mppi_reduce(egg_batch* b, const double* u_d, int horizon, const double* cost_d, const double* baseline_d,
                    double lambda, double* out_d);

/* CEM (cross-entropy method, INTEGRATION.md): sample around a mean schedule with a per-step standard
 * deviation, keep the k cheapest rollouts (the elites) and refit mean and standard deviation to them.
 *
 * u_d[t][w][b][j] = clamp(mean_d[t][b][j] + std_d[t][b][j] eps, u_lo[b][j], u_hi[b][j]) for t < horizon
 * and every local world w; mean_d and std_d are DEVICE [horizon][n_bodies][6] arrays, u_d is
 * [horizon][W][n_bodies][6].  eps is exactly the eps of egg_sample_controls for the same seed,
 * iteration and global world first + w (the same Philox key and counter, uniforms and Box-Muller), so
 * with std_d[t] = sigma for every t the output is that of egg_sample_controls bit for bit.  Global
 * world 0 and std = 0 keep clamp(mean) bit for bit.  The bounds come from egg_set_sampler; its sigma is
 * not used.  std_d values are the caller's: finite and >= 0 give a clamped normal sample.
 * EGG_ERR_STATE without a sampler or before egg_init; EGG_ERR_ARG for horizon < 1, first < 0, a
 * pointer that is not device memory of the batch's device, or one that is not 16-byte aligned.
 * Asynchronous on the batch stream; one launch. */
int egg_sample_controls_std(egg_batch* b, const double* mean_d, const double* std_d, int horizon, unsigned long long seed,
                            unsigned long long iteration, int first, double* u_d);

/* out_d[i] ([k][horizon][n_bodies][6], device) = the schedule of local world worlds[i] in u_d
 * ([horizon][W][n_bodies][6]), copied bit for bit.  worlds is a HOST int array, each entry in [0, W),
 * duplicates allowed; 1 <= k <= W (the rules of egg_gather_state).  EGG_ERR_ARG for those, horizon < 1
 * or a pointer that is not device memory of the batch's device; EGG_ERR_STATE before egg_init.
 * Asynchronous on the batch stream; one launch. */
int egg_gather_controls(egg_batch* b, const double* u_d, int horizon, const int* worlds, int k, double* out_d);

/* The moments of k schedules rows_d [k][horizon][n_bodies][6] (device), per element:
 * out_d[0] = mean = (the rows added in row order) / k and out_d[1] = the population standard
 * deviation sqrt(sum_i (x_i - mean)^2 / k), a second pass in row order with every square rounded
 * before it is added; out_d is [2][horizon][n_bodies][6] (device).  No atomics: the bits depend only
 * on k, n_bodies, horizon and the rows, and NaN propagates.  EGG_ERR_ARG for k < 1, horizon < 1 or a
 * pointer that is not device memory of the batch's device; EGG_ERR_STATE before egg_init.
 * Asynchronous on the batch stream; one launch. */
int egg_control_moments(egg_batch* b, const double* rows_d, int k, int horizon, double* out_d);

/* Ensemble::UpdateContacts + CheckAndCorrectEnsembleState only (ensembles.cc:445-480, 241-329):
 * runs the narrowphase kernel on the current state without stepping; read the result with
 * egg_get_contacts / egg_get_pair_hits. */
int egg_update_contacts(egg_batch* b);

/* Ensemble::M_inverse() / external_force_torque_ taps (ensembles.h:68,88-89) as frozen by egg_init:
 * minv_lin [W][n], minv_ang [W][n][9], f_ext [W][n][6].  Any pointer may be NULL. */
int egg_get_static(egg_batch* b, double* minv_lin, double* minv_ang, double* f_ext);

/* Device-side copy of the dynamic Body state (p,R,v,w of every world): egg_snapshot saves it,
 * egg_restore puts it back (asynchronous on the batch stream).  Used to replay a step from the
 * same state (stepwise parity, stationary benchmarks, MPC rollouts from a common start). */
int egg_snapshot(egg_batch* b);
int egg_restore(egg_batch* b);

/* Reads back Body state (body.h:50-58 accessors); synchronises the stream. */
int egg_get_bodies(egg_batch* b, double* p, double* R, double* v, double* w);

/* Parity taps of the last step: the surviving contact list in reference order (ensembles.cc:445-480
 * after :241-329), its multipliers and per-row state.  Any pointer may be NULL.  Layouts:
 * count[W]; i0,i1,code [W][max_contacts]; pos,nrm [W][max_contacts][3]; depth [W][max_contacts];
 * lambda [W][3*(n_joints+max_contacts)] in row order (joints first, ensembles.cc:234-239);
 * row_state same shape: 0 free, 1 at lower bound, 2 at upper bound, 3 equality row. */
int egg_get_contacts(egg_batch* b, int* count, int* i0, int* i1, double* pos, double* nrm,
                     double* depth, int* code, double* lambda, int* row_state);

/* The same taps for the worlds [first, first + n_worlds) only: arrays are sized for n_worlds worlds.
 * Use this for spot checks of large batches (egg_get_contacts of 65536 x 64-body worlds moves GBs). */
int egg_get_contacts_range(egg_batch* b, int first, int n_worlds, int* count, int* i0, int* i1, double* pos,
                           double* nrm, double* depth, int* code, double* lambda, int* row_state);

/* Colliding pairs of the last step in (i<j) lexicographic order with CollisionInfo.code and the
 * pre-de-dup contact count (requires desc.taps = 1).  n_hits[W]; pi,pj,code,count [W][max_pairs]. */
int egg_get_pair_hits(egg_batch* b, int* n_hits, int* pi, int* pj, int* code, int* count, int max_pairs);
int egg_get_pair_hits_range(egg_batch* b, int first, int n_worlds, int* n_hits, int* pi, int* pj, int* code, int* count, int max_pairs);

/* status[W] (egg_status bits); stats [W][8] = {n_contacts_raw, n_contacts, n_rows, n_pair_hits,
 * sweeps, pivots, cfm_applied, reserved}; residual[W] = last GetResidualError. */
int egg_get_status(egg_batch* b, int* status, int* stats, double* residual);

/* Dense solver only: FP64 operations the reference algorithm spends on each world's last solve
 * (flops[W]; multiplications and additions counted separately): one factorisation for the cfm
 * decision, the LU inverse and products of the Schur complement (lcp.cc:286-294), and per Murty
 * pivot one LDL^T of the basic block, its two triangular solves and w = A_NS x_S (lcp.cc:195-232).
 * Feeds the FP64 roofline of bench.py --workload c4. */
int egg_get_dense_work(egg_batch* b, double* flops);

/* Development aid: 32 device-side counters (phase cycle counts of the dense kernel when the
 * library is built with EGG_DENSE_TIMING=1, zeros otherwise); reset != 0 clears them. */
int egg_get_debug_counters(egg_batch* b, unsigned long long* out32, int reset);

/* MPC rollout cost per world written to a DEVICE buffer of n_worlds doubles (feeds the NCCL
 * allgather): cost = -(x_body0 - x0_body0) + 10 (z_body0 - z0_body0)^2 with (x0,z0) the pose at
 * egg_init.  The reference has no cost function; this definition is ours (SURVEY.md §8d C5).
 * A configurable cost accumulated over the horizon: egg_set_cost / egg_step_controlled_cost. */
int egg_rollout_costs(egg_batch* b, double* cost_d);

/* Stream plumbing: run the batch on a caller-owned cudaStream_t (e.g. torch's current stream) so
 * that caller-side CUDA events bracket the kernels. */
int egg_set_stream(egg_batch* b, void* cuda_stream);
int egg_sync(egg_batch* b);

/* Per-world contact capacity actually allocated (max_contacts after rounding / the automatic rule). */
int egg_capacity(const egg_batch* b);

/* Which kernel instances the batch runs (read-only, no device access).  out[0] lanes per world of
 * the PGS group stream (0 for the other solvers), out[1] worlds per warp (32 / out[0], or 0),
 * out[2] M^-1 layout of the PGS kernel: 0 general 3x3, 1 isotropic per body, 2 isotropic and
 * uniform, -1 before the first step after egg_init decides it, out[3] constraint-record format:
 * 0 per-world records (dense, Jacobi, SOR), 1 PGS group stream, 2 PGS run format, -1 for PGS before
 * the first step after egg_init, out[4] runs per world and stage of the run format (0 without it),
 * out[5] record precision (64 or 32), out[6] narrowphase threads per world, out[7] record-assembly
 * threads per world (for the run format: after the first step).  The development overrides
 * EGG_PGS_LPW, EGG_PGS_MIN_WARPS_PER_SM, EGG_PGS_RUNS, EGG_PGS_RUN_CAP, EGG_PGS_TARGET_CTAS,
 * EGG_COLLIDE_NT, EGG_RECORDS_NT (and EGG_PGS_CTAS_PER_SM, EGG_PGS_PF) are read by egg_create and
 * apply to that batch only. */
int egg_get_kernel_config(const egg_batch* b, int out[8]);

/* Bytes of device memory held by the batch; number of kernel launches issued so far. */
long long egg_device_bytes(const egg_batch* b);
long long egg_launch_count(const egg_batch* b);

/* Per-kernel device time.  With profiling on, egg_step brackets each of its kernels with CUDA
 * events on the batch stream; egg_get_kernel_ms synchronises and returns the milliseconds
 * accumulated since the last call: out[0] narrowphase, out[1] row assembly, out[2] solve +
 * integrate, out[3] = number of steps counted. */
int egg_set_profiling(egg_batch* b, int on);
int egg_get_kernel_ms(egg_batch* b, double* out4);

/* FP64 roofline denominator: a dependent-free DFMA loop on every SM of `device`; returns TFLOP/s
 * (2 flop per FMA), or a negative egg_error. */
double egg_fp64_peak_tflops(int device);

/* Pinned host staging (cudaHostAlloc) for end-to-end measurements. */
void* egg_host_alloc(long long bytes);
void egg_host_free(void* p);

const char* egg_last_error(void);
const char* egg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* EGG_CUDA_H_ */
