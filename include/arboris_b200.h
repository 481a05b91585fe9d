/* arboris_b200 -- C ABI of the B200-native batched Arboris simulation step.
 *
 * The reference (sbarthelemy/arboris-python) has no FFI: its "plugin API" is a
 * set of Python classes (arboris/core.py:158-339) and the four World methods
 * that make one time step (arboris/core.py:682-980, driven by simulate(),
 * core.py:1334-1365).  This header is the C boundary a binding of that API sits
 * on: plain pointers and sizes, no C++/torch types, every call returns an int
 * (0 = ok, <0 = error, text via arb_last_error()) and never throws.
 *
 * Conventions
 *  - All arithmetic is IEEE fp64.  Twists are [angular; linear]; 4x4 matrices
 *    are row-major; H_ab maps b-coordinates to a-coordinates.
 *  - A *model* is the immutable flattened tree (what World.init(), core.py:608-635,
 *    and the constructors of joints/constraints/controllers fix).  Body 0 is the
 *    ground; body j+1 is the child of joint j; joints are in the reference's
 *    depth-first order (core.py:416-419), which also numbers the dofs.
 *  - A *batch* is W independent worlds of one model on one CUDA device.  State is
 *    CALLER-OWNED device memory, structure-of-arrays with the world index
 *    fastest:  gpos[ngpos][W], gvel[ndof][W], cforce[nrows][W].
 *      gpos  : per joint, 16 doubles (row-major 4x4) for FreeJoint, else its
 *              ndof angles/translations            (Joint.gpos, core.py:227-240,
 *                                                   joints.py:13-33)
 *      gvel  : World._gvel                          (core.py:626-629)
 *      cforce: every constraint's _force, stacked in registration order
 *              (constraints.py:52,153,422); only BallAndSocketConstraint rows
 *              are read as state (warm start), the others are outputs (the host-buffer
 *              entry points copy cforce host -> device only for models with such rows).
 *  - All work is enqueued on the batch's stream and is asynchronous w.r.t. the
 *    host unless stated.  One batch is driven by one host thread at a time.
 */
#ifndef ARBORIS_B200_H
#define ARBORIS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* joints.py: FreeJoint:10, RzRyRxJoint:59, RzRyJoint:107, RzRxJoint:149,
 * RyRxJoint:188, RzJoint:227, RyJoint:305, RxJoint:328, TxTyTzJoint:352 */
typedef enum {
  ARB_JOINT_FREE = 0, ARB_JOINT_RZRYRX = 1, ARB_JOINT_RZRY = 2, ARB_JOINT_RZRX = 3,
  ARB_JOINT_RYRX = 4, ARB_JOINT_RZ = 5, ARB_JOINT_RY = 6, ARB_JOINT_RX = 7,
  ARB_JOINT_TXTYTZ = 8
} arb_joint_type;

/* constraints.py: JointLimits:15, BallAndSocketConstraint:92,
 * SoftFingerContact:300 over plane_point_collision (collisions.py:105) */
typedef enum {
  ARB_CONS_JOINT_LIMITS = 0, ARB_CONS_BALL_SOCKET = 1, ARB_CONS_SOFT_FINGER_PLANE_POINT = 2
} arb_constraint_type;
/* shape pair of a SoftFingerContact, ordered as collisions.choose_solver (collisions.py:14-65)
 * orders it; a Point is a sphere of radius 0 */
typedef enum {
  ARB_PAIR_PLANE_SPHERE = 0,    /* plane_sphere_collision / plane_point_collision (:95-111) */
  ARB_PAIR_SPHERE_SPHERE = 1,   /* sphere_sphere_collision / sphere_point_collision (:67-85) */
  ARB_PAIR_BOX_SPHERE = 2       /* box_sphere_collision (:87-93) */
} arb_contact_pair;

/* controllers.py: WeightController:10, ProportionalDerivativeController:63 */
typedef enum { ARB_CTRL_WEIGHT = 0, ARB_CTRL_PD = 1 } arb_controller_type;

#define ARB_CONS_NINT 4
#define ARB_CONS_NDBL 48
#define ARB_GS_SWEEPS 20          /* core.py:930 */

/* Flattened model; every pointer is HOST memory, copied by arb_model_create.
 *  cons_int[c] / cons_dbl[c]:
 *   JOINT_LIMITS : int {joint, dof, gpos index, enabled}; dbl {min, max, proximity}
 *   BALL_SOCKET  : int {body0, body1, -, enabled}; dbl {bpose0[16], bpose1[16]}
 *   SOFT_FINGER  : int {body of shape 0, body of shape 1, arb_contact_pair, enabled};
 *                  dbl {shape 0 frame bpose[16], shape 1 frame bpose[16],
 *                       plane coeffs[4] or box half extents[3] @32, mu @36, eps[3] @37,
 *                       proximity @40, radius of shape 0 @41, radius of shape 1 @42}
 *  ctrl_int[a] / ctrl_dbl[a]:
 *   WEIGHT : dbl {gravity}
 *   PD     : int {m, blob offset}; blob {dof map[m], gpos map[m], kp[m*m],
 *            kd[m*m], gpos_des[m], gvel_des[m]} (maps stored as doubles)      */
typedef struct arb_model_desc {
  int32_t ndof, ngpos, njoints, nconstraints, ncontrollers, nrows, nblob;
  const int32_t *joint_type, *joint_parent, *joint_dof, *joint_gpos;   /* [njoints] */
  const double *joint_Hpr, *joint_Hcn;      /* [njoints][16] Joint._frame0/1 .bpose, core.py:1295-1296 */
  const double *body_mass, *body_visc;      /* [njoints][36] Body.mass/.viscosity, core.py:1071-1072 */
  const int32_t *cons_type;                 /* [nconstraints] */
  const int32_t *cons_int;                  /* [nconstraints][ARB_CONS_NINT] */
  const double *cons_dbl;                   /* [nconstraints][ARB_CONS_NDBL] */
  const int32_t *cons_row;                  /* [nconstraints] first row in cforce */
  const int32_t *ctrl_type;                 /* [ncontrollers] */
  const int32_t *ctrl_int;                  /* [ncontrollers][4] */
  const double *ctrl_dbl;                   /* [ncontrollers][4] */
  const double *ctrl_blob;                  /* [nblob] */
  double up[3];                             /* World._up, core.py:351 */
} arb_model_desc;

typedef struct arb_model arb_model;
typedef struct arb_batch arb_batch;

/* which-selectors for the read-backs */
typedef enum {            /* World properties core.py:645-655, 754-761 */
  ARB_MASS = 0, ARB_NLEFFECTS = 1, ARB_VISCOSITY = 2, ARB_IMPEDANCE = 3, ARB_ADMITTANCE = 4
} arb_matrix_id;
typedef enum {            /* Body attributes core.py:1107-1125 */
  ARB_BODY_POSE = 0,      /* 16 doubles */
  ARB_BODY_TWIST = 1,     /* 6 */
  ARB_BODY_JAC = 2,       /* 6 x ndof, row-major */
  ARB_BODY_DJAC = 3,      /* 6 x ndof */
  ARB_BODY_NLE = 4        /* 36 */
} arb_body_id;
typedef enum {
  ARB_CONS_ACTIVE = 0,    /* int32 [nconstraints]  Constraint.is_active() */
  ARB_CONS_BRANCH = 1,    /* int32 [nconstraints]  branch taken by the last solve(): soft finger
                             1 separating / 2 static / 3 sliding (constraints.py:781,799,803);
                             joint limits 1 free / 2 min / 3 max (constraints.py:77,81,85) */
  ARB_CONS_SDIST = 2,     /* double [nconstraints] PointContact._sdist */
  ARB_CONS_ZIDX = 3       /* int32 [nconstraints][3] argsort(|normal|) used by zaligned,
                             homogeneousmatrix.py:225 (index work, bit-exact) */
} arb_constraint_id;
typedef enum { ARB_VEC_GFORCE = 0 } arb_vector_id;   /* World._gforce, core.py:665-667 */

/* per-world status bits (arb_batch_status) */
#define ARB_STATUS_NONFINITE   1   /* NaN/Inf in gvel or gpos */
#define ARB_STATUS_SINGULAR    2   /* zero pivot inverting the impedance (LinAlgError in the reference) */
#define ARB_STATUS_EIG_NOROOT  4   /* sliding solve found no real eigenvalue <= 0: s = -1e10 (constraints.py:827-830) */
#define ARB_STATUS_EIG_NOCONV  8   /* QR iteration hit its cap */

const char *arb_last_error(void);
int arb_version(void);

/* replaces: World.init() + object constructors (core.py:608-635) */
int arb_model_create(const arb_model_desc *desc, arb_model **out);
void arb_model_destroy(arb_model *model);

/* W worlds of `model` on CUDA device `device`; `stream` is a cudaStream_t (NULL =
 * default stream).  Scratch is owned by the library. */
int arb_batch_create(const arb_model *model, int64_t nworlds, int device, void *stream,
                     arb_batch **out);
void arb_batch_destroy(arb_batch *batch);
int arb_batch_set_stream(arb_batch *batch, void *stream);
/* tuning/testing switches:
 *  "force_phases" 1: arb_step runs the four API phase kernels instead of the fused stages;
 *  "sort_period"  N: the fused step re-assigns the worlds to threads by contact state every N
 *                 steps (default 2; 0: never, worlds stay in arrival order); results are
 *                 bit-identical whatever the value;
 *  "gs_stage"     1 (default): the Gauss-Seidel kernel finds the operands of a contact visit (the
 *                 4x4 Delassus block, its pseudo-inverse, the contact map, sdist) in shared memory,
 *                 copied there one visit ahead by TMA bulk copies (models of at most 32
 *                 constraints; larger ones run the other kernel); 0: the kernel that loads them
 *                 from global memory; bit-identical results;
 *  "gs_plain"     0 (before the batch's first step): the staged kernel's general instantiation even
 *                 for a model that qualifies for the plain one (joint limits and one-body contacts of
 *                 contact-aligned bodies only); bit-identical results, a test switch;
 *  "gs_coop"      1: block-cooperative Gauss-Seidel kernel (sliding solves pooled through
 *                 shared memory) instead of the per-lane one; bit-identical results;
 *  "prepare_group" 1: the prepare stage runs with a group of 16 lanes per world and the world's
 *                 intermediates in shared memory (csrc/arb_group.cuh), the finish stage as
 *                 q'+ = q_free + K y; same results to 1e-10 (other summation order), 5x slower than the
 *                 default lane-per-world stages on human36 (DESIGN.md 3.4): an A/B switch; it does not
 *                 support applied forces (arb_batch_bind_applied_forces);
 *  "time_stages"  1: CUDA events around every fused stage, synchronising after every step -- a
 *                 diagnostic for bench.py, read with arb_batch_stage_ms; setting it clears the
 *                 accumulators */
int arb_batch_set_option(arb_batch *batch, const char *name, int value);

/* caller-owned DEVICE state, layouts in the header comment */
int arb_batch_bind_state(arb_batch *batch, double *gpos, double *gvel, double *cforce);

/* Per-world parameters of the ProportionalDerivativeControllers (controllers.py:63-159: kp, kd,
 * gpos_des, gvel_des; used at :141-159).  The reference keeps them on the controller object of ONE
 * world; a batch may give every world its own.  DEVICE arrays [npd][W], world index fastest, caller-
 * owned like the state; row p belongs to the p-th controlled dof, counting the controllers in
 * registration order and each controller's dofs in its own order (arb_model_pd_dofs lists them).
 * kp / kd rows are the DIAGONAL gains of that dof (off-diagonal gains stay the model's).  A NULL
 * pointer means "the model's value for every world"; all NULL unbinds.  Read by every later
 * arb_update_controllers / arb_step. */
int arb_batch_bind_controller_params(arb_batch *batch, const double *kp, const double *kd,
                                     const double *gpos_des, const double *gvel_des);
/* dof of each row of those arrays: writes min(npd, cap) entries, returns npd (dofs may be NULL) */
int arb_model_pd_dofs(const arb_model *model, int32_t *dofs, int cap);
/* Per-world applied forces: what a reference Controller whose update() returns (gforce, 0) adds,
 * as one such controller registered AFTER the model's ones, with no impedance term.
 *  gforce : DEVICE [ndof][W] generalized forces, added to World._gforce (core.py:811-818).
 *  wrench : DEVICE [nbodies][6][W] wrenches [torque; force] in GROUND axes acting at the origin of
 *           the frame of body bodies[i]; the step adds J_b^T [R_b^T torque; R_b^T force], with J_b the
 *           body Jacobian in the body frame (core.py:1171-1176) and R_b the body's rotation at the
 *           start of the step.
 *  bodies : HOST list of nbodies distinct body indices 1..njoints (as in arb_get_body; the ground
 *           is refused), copied into a table of the batch.
 * Both arrays are caller-owned like the state, world index fastest, and read (by WORLD index,
 * whatever the thread assignment) at every step of arb_update_controllers, arb_step and
 * arb_step_begin: write them in place, in stream order, to change the forces between calls.
 * A NULL pointer or nbodies = 0 means no such force; all NULL / 0 unbinds.  -1 for a body out of
 * range, the ground, a duplicate body or a wrench without bodies (the previous binding is kept).
 * The "prepare_group" option does not support them: arb_step / arb_step_begin return -1 while
 * both are set. */
int arb_batch_bind_applied_forces(arb_batch *batch, const double *gforce, int nbodies, const int32_t *bodies,
                                  const double *wrench);
/* which implementation arb_step runs for this batch: 1 = the fused stages, 0 = the four phase
 * kernels (a PD controller with off-diagonal gains or two controllers on one dof -- Z then has
 * entries the per-dof articulated elimination does not fold -- or the "force_phases" option).
 * *why (may be NULL) receives a static string naming the reason. */
int arb_batch_step_path(const arb_batch *batch, const char **why);

/* replaces World.update_dynamic (core.py:682-734; Body.update_dynamic :1272-1315) */
int arb_update_dynamic(arb_batch *batch);
/* replaces World.update_controllers (core.py:811-818) */
int arb_update_controllers(arb_batch *batch, double dt);
/* replaces World.update_constraints (core.py:910-937) */
int arb_update_constraints(arb_batch *batch, double dt);
/* replaces World.integrate (core.py:974-980) */
int arb_integrate(arb_batch *batch, double dt);
/* replaces the simulate() loop body (core.py:1356-1363) for nsteps consecutive steps
 * of length dts[i] (HOST array); intermediate matrices stay on chip */
int arb_step(arb_batch *batch, const double *dts, int nsteps);
/* the same step in two halves, for callers that observe the world between
 * update_constraints and integrate like the reference's Observer.update (core.py:1360-1362):
 * arb_step_begin = update_dynamic + update_controllers + update_constraints (state untouched,
 * constraint forces written), arb_step_end = integrate.  Between the two, arb_get_body
 * (POSE, TWIST) and arb_get_constraint read the step's quantities. */
int arb_step_begin(arb_batch *batch, double dt);
int arb_step_end(arb_batch *batch, double dt);
/* same, with HOST state buffers (same layouts): H2D, nsteps, D2H, synchronous */
int arb_step_host(arb_batch *batch, double *h_gpos, double *h_gvel, double *h_cforce,
                  const double *dts, int nsteps);

/* same for a SLICE of a larger host array: row e of the host arrays starts at h_x + e*host_ld
 * (host_ld >= nworlds, in worlds), so that several batches -- each on its own stream -- can work on
 * column blocks of one [elem][W_total] host state and overlap their copies with each other's
 * kernels.  synchronize = 0: returns with the work enqueued; see arb_batch_synchronize. */
int arb_step_host_strided(arb_batch *batch, double *h_gpos, double *h_gvel, double *h_cforce,
                          int64_t host_ld, const double *dts, int nsteps, int synchronize);
/* wait for everything enqueued on the batch's stream */
int arb_batch_synchronize(arb_batch *batch);
/* the two copies of arb_step_host_strided alone, on a stream of the caller's choice (cudaStream_t):
 * to_device != 0: host slice -> the batch's bound state arrays; 0: the reverse.  Lets a caller keep
 * the kernels of all column blocks on ONE stream (one kernel on the GPU at a time) and the copies on
 * two others, ordered by events (batch.HostPipeline, mode "serial").  Same state arrays as
 * World._gvel / Joint.gpos in the reference (core.py:626-629). */
int arb_state_copy_host_strided(arb_batch *batch, double *h_gpos, double *h_gvel, double *h_cforce,
                                int64_t host_ld, int to_device, void *stream);

/* read-backs into DEVICE buffers, worlds [w0, w1), world-major: out[w-w0][...] */
int arb_get_matrix(arb_batch *batch, int which, double *out, int64_t w0, int64_t w1);
int arb_get_vector(arb_batch *batch, int which, double *out, int64_t w0, int64_t w1);
int arb_get_body(arb_batch *batch, int which, int body, double *out, int64_t w0, int64_t w1);
int arb_get_constraint(arb_batch *batch, int which, void *out, int64_t w0, int64_t w1);
/* int32 flags[W] (DEVICE), bits ARB_STATUS_*, accumulated since the last call */
int arb_batch_status(arb_batch *batch, int32_t *flags);

/* counters for bench.py: kernels launched by this library since batch creation */
int64_t arb_batch_launch_count(const arb_batch *batch);
/* accumulated device milliseconds of the fused stages since "time_stages" was set:
 * out4 = {prepare, gs, finish, number of steps timed} */
int arb_batch_stage_ms(const arb_batch *batch, double *out4);
/* measured fp64 FMA throughput of the device in flop/s (DFMA micro-benchmark, about 50 ms) */
int arb_measure_fp64_peak(int device, double *flops_per_s);

#ifdef __cplusplus
}
#endif
#endif /* ARBORIS_B200_H */
