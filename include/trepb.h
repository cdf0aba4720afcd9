/* trepb.h — C ABI of the B200-native batched MidpointVI library (libtrepb.so).
 *
 * Drop-in boundary for ONE path of MurpheyLab/trep: the midpoint variational integrator's
 * DEL step and its linearization, evaluated over a batch of independent instances.
 * Plain C, plain pointers and sizes, no Python and no torch types.
 *
 * What each entry point replaces in the reference (paths relative to the reference root):
 *
 *   trepb_system_create      the "synchronize" product of trep/system.py:672-840 +
 *                            trep/frame.py:658-721 (frame order, config_gen, cache_index,
 *                            masses) and the plugin structs of trep/_trep/trep.h:305-375,
 *                            flattened (see trepb_sysdesc).
 *   trepb_step_batch*        _trep._MidpointVI._solve_DEL  == MidpointVI_solve_DEL
 *                            (trep/_trep/midpointvi.c:691-747, exported as C-API slot
 *                            capi_MidpointVI_solve_DEL, trep/_trep/c_api.h:88,693), looped
 *                            the way MidpointVI.step does (trep/midpointvi.py:174-201):
 *                            q1<-q2, p1<-p2, kinematic part of q2 <- k2, Newton start = q1.
 *   trepb_calc_p2_batch*     _MidpointVI.calc_p2 (trep/_trep/midpointvi.c:491-504,2702-2708),
 *                            i.e. MidpointVI.initialize_from_configs (midpointvi.py:155-172).
 *   trepb_deriv2_batch*      _MidpointVI._calc_deriv2 (trep/_trep/midpointvi.c:2516-2545): the
 *                            second-derivative tensors q2/p2/lambda1 _d{q1,p1,u1,k2}d{q1,p1,u1,k2}.
 *   trepb_project_batch*     DSystem.project / DOptimizer.armijo_simulate: closed-loop rollouts
 *                            (trep/discopt/dsystem.py:426-457, doptimizer.py:405-428).
 *   trepb_lqr_batch*         discopt.dlqr.solve_tv_lqr (trep/discopt/dlqr.py:9-38), the Riccati sweep of
 *                            DSystem.calc_feedback_controller (trep/discopt/dsystem.py:474-494).
 *   trepb_tangent_batch*     DSystem.dproject (trep/discopt/dsystem.py:460-471): the forward sweep of a
 *                            descent direction, on the slabs the two calls above leave in HBM.
 *   trepb_adjoint_batch*     the costate recursion of DOptimizer.calc_newton_model
 *                            (trep/discopt/doptimizer.py:319-345).
 *   trepb_track_batch*       DCost (trep/discopt/dcost.py) summed as DOptimizer.calc_cost / calc_dcost, and the
 *                            LQ model of DOptimizer's steepest / quasi / newton directions.
 *   trepb_candidates_batch*  the step-size candidates of DOptimizer.armijo_search.
 *   trepb_dare_batch*        no counterpart: the stationary LQR gain at an equilibrium, which a user of the
 *                            reference computes on the host with scipy.linalg.solve_discrete_are.
 *   trepb_dlyap_batch*       no counterpart: closed-loop cost and stability of stationary gains under a batch of
 *                            models, which a user computes on the host with scipy.linalg.solve_discrete_lyapunov.
 *   trepb_linearize_batch*  DSystem.set + fdx + fdu for every k of
 *                            DSystem.linearize_trajectory (trep/discopt/dsystem.py:229-250,
 *                            284-317, 406-423) == solve_DEL + MidpointVI_calc_deriv1
 *                            (trep/_trep/midpointvi.c:1100-1120).
 *   status[] / iters[]       the reference's exceptions (ConvergenceError midpointvi.c:715-718,
 *                            singular LU math-code.c:393-398) become per-instance codes; the
 *                            batch is never aborted.
 *
 * All matrices are row-major doubles.  Per-instance arrays are packed instance-major
 * ("[B][n]"): instance b's vector starts at ptr + b*n.
 *
 * `_dev` entry points take DEVICE pointers (inputs already resident in HBM) and enqueue on
 * `stream` (a cudaStream_t passed as void*; NULL = default stream) without synchronizing.
 * One handle may be used from several host threads and on several streams: launches that need
 * scratch memory owned by the handle (the table-driven thread kernels' workspace slab, the
 * second-derivative passes) are ordered on the device behind the previous such launch, whatever
 * stream that one used; the specialised and the cooperative step / linearize / project kernels own
 * no scratch and overlap freely.  trepb_last_kernel_ms refers to the handle's most recent launch.
 * After a failed step of a rollout (status != 0) the `_dev` entry points leave the rows of X / U /
 * traj_q / traj_p past the failure untouched (the caller's memory); the host-pointer entry points
 * return zeros there.
 * The un-suffixed entry points take HOST pointers, copy in, run, copy out and synchronize.
 *
 * Every function returns 0 on success, non-zero on failure; trepb_last_error() describes
 * the failure.  There is no CPU fallback: without a CUDA device every compute entry point
 * fails with TREPB_ERR_CUDA.
 */
#ifndef TREPB_H
#define TREPB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TREPB_ABI_VERSION 2   /* 2: times[] in step / project args, traj_len in lin args, calc_f / discrete_fm2,
                                   trepb_comm_* / trepb_ipc_* (appended fields and new entry points only) */

/* error codes */
#define TREPB_OK 0
#define TREPB_ERR_INVALID 1   /* bad description / arguments */
#define TREPB_ERR_CUDA 2      /* CUDA runtime / no device */
#define TREPB_ERR_COMPILE 3   /* reserved */
#define TREPB_ERR_UNSUPPORTED 4

/* frame transform kinds (trep/_trep/trep.h:168-273) */
#define TREPB_WORLD 0
#define TREPB_TX 1
#define TREPB_TY 2
#define TREPB_TZ 3
#define TREPB_RX 4
#define TREPB_RY 5
#define TREPB_RZ 6
#define TREPB_CONST_SE3 7

/* potential / force / constraint kinds: the built-in C plugin kinds on the path */
#define TREPB_POT_GRAVITY 0        /* d = gx gy gz                       potentials/gravity.c      */
#define TREPB_POT_LINEAR_SPRING 1  /* i = frame1 frame2 ; d = k x0       potentials/linearspring.c */
#define TREPB_POT_CONFIG_SPRING 2  /* i = config        ; d = k q0       potentials/configspring.c */
#define TREPB_POT_NONLINEAR_CONFIG_SPRING 3 /* i = config, dpool offset, n x-points ; d = m b ; dpool: x[n], coeffs[n-1][6]
                                             potentials/nonlinear_config_spring.c + spline.c */
#define TREPB_FORCE_DAMPING 0      /* i = dpool offset, nd ; coefficients per dyn config  forces/damping.c */
#define TREPB_FORCE_CONFIG 1       /* i = config input                   forces/configforce.c      */
#define TREPB_FORCE_LINEAR_DAMPER 2/* i = ipool offset, npath ; d = c    forces/lineardamper.c     */
#define TREPB_CON_DISTANCE 0       /* i = frame1 frame2 config|-1 ; d = distance tolerance  constraints/distance.c */
#define TREPB_CON_POINT1D 1        /* i = frame1 frame2 component ; d = - tolerance         constraints/point.c    */
#define TREPB_CON_PLANE 2          /* i = plane_frame point_frame ; d = n0 tolerance n1 n2  constraints/plane.c    */
/* wrenches: i = frame, ipool offset of six input indices (-1: constant component), dpool offset of the six
 * constants                                                         forces/{body,hybrid,spatial}wrench.c */
#define TREPB_FORCE_BODY_WRENCH 3
#define TREPB_FORCE_HYBRID_WRENCH 4
#define TREPB_FORCE_SPATIAL_WRENCH 5

/* Flattened system.  Frame 0 is the world frame; frames are in pre-order (parent before child),
 * configs are [dynamic..., kinematic...].  Arrays are only read during trepb_system_create. */
typedef struct trepb_sysdesc {
    int32_t n_frames, nd, nk, nu;
    int32_t n_potentials, n_forces, n_constraints;
    int32_t n_ipool, n_dpool, _pad;
    const int32_t* frame_parent;  /* [n_frames]      -1 for world                       */
    const int32_t* frame_kind;    /* [n_frames]      TREPB_TX ...                       */
    const int32_t* frame_config;  /* [n_frames]      driving config or -1               */
    const double*  frame_value;   /* [n_frames]      constant transform parameter       */
    const double*  frame_se3;     /* [n_frames][12]  row-major [R|p] for CONST_SE3      */
    const double*  frame_mass;    /* [n_frames][4]   m Ixx Iyy Izz                      */
    const int32_t* pot_kind;   const int32_t* pot_i;   const double* pot_d;    /* [n][1],[n][4],[n][4] */
    const int32_t* force_kind; const int32_t* force_i; const double* force_d;
    const int32_t* con_kind;   const int32_t* con_i;   const double* con_d;
    const int32_t* ipool;      const double* dpool;
} trepb_sysdesc;

typedef struct trepb_system trepb_system; /* opaque */

/* flags for trepb_system_create */
#define TREPB_FLAG_NO_SPECIALIZE 1  /* use the table-driven general kernels even for small systems */
#define TREPB_FLAG_NO_COOP 2        /* table-driven systems: always one thread per instance */
#define TREPB_FLAG_FORCE_COOP 4     /* table-driven systems: always the cooperative kernels (one or two warps per
                                       instance, workspace in shared memory); fails if they do not apply */
#define TREPB_FLAG_D2_PAIRWISE 8    /* table-driven systems: second derivatives by one hyper-dual residual
                                       evaluation per parameter pair (the scheme the small specialised
                                       systems use) instead of one dual evaluation of the Jacobian tables
                                       per parameter followed by a contraction */

/* Cooperative kernels, shapes built in several flavours (the marionette's).  The default is the one with the highest
 * throughput on full batches: one warp per instance with part of the first-derivative workspace in an L2-resident
 * slab of global memory (16 instances per SM, name ".../ext"). */
#define TREPB_FLAG_COOP_ONE_WARP 32  /* one warp per instance, the whole workspace in shared memory (8 per SM) */
#define TREPB_FLAG_COOP_TWO_WARPS 64 /* two warps per instance (8 per SM): the lowest latency per linearization on
                                       batches that do not fill the GPU (name ".../pair") */
#define TREPB_FLAG_NO_LITERAL 16     /* specialised systems: skip an all-literal instantiation built for exactly this
                                       description and use the run-time-parameter kernel of its structure */
#define TREPB_FLAG_COOP_VARIED 128   /* cooperative handles: the *_varied_batch* entry points run on the varied
                                       cooperative kernels of the handle's flavour instead of being refused; plain
                                       calls are unchanged.  Ignored on other handles.  See "per-instance physical
                                       parameters" below. */

/* Loads a plug-in built by trep_b200/build.py:build_plugin from a system description: ahead-of-time specialised
 * (register-resident) kernels for a structure the library was not built with - the role the reference gives to
 * compiling a system's own C plugins.  *n_added (may be NULL) receives the number of kernel sets registered;
 * a library that registers none (not a plug-in, or loaded before) is TREPB_ERR_INVALID.  trepb_system_create
 * then matches the structure like a built-in one (parameters stay run-time data).                           */
int  trepb_load_plugin(const char* path, int* n_added);

int  trepb_abi_version(void);
const char* trepb_last_error(void);

/* Validate + flatten + upload tables to `device`.  If the description's structure (trepb_struct_hash)
 * matches one of the systems specialised ahead of time (generated constexpr structure, fully unrolled,
 * register-resident, parameters at run time; see trepb_codegen) that kernel set is used, otherwise the table-driven
 * kernels: one thread per instance for small systems, the cooperative kernels (one warp per
 * instance, link tables and workspace in shared memory) when the per-instance workspace is too
 * large to stay on chip (e.g. the marionette). */
int  trepb_system_create(const trepb_sysdesc* desc, int device, int flags, trepb_system** out);
void trepb_system_destroy(trepb_system* sys);
int  trepb_system_dims(const trepb_system* sys, int32_t* nq, int32_t* nd, int32_t* nk,
                       int32_t* nu, int32_t* nc);
/* 1 if a specialised (compile-time frame tree) kernel is in use, 0 if table-driven. */
int  trepb_system_is_specialized(const trepb_system* sys);
const char* trepb_system_kernel_name(const trepb_system* sys);
/* 1 if the cooperative kernels (one warp per instance, shared-memory workspace) are in use. */
int  trepb_system_is_cooperative(const trepb_system* sys);
/* Launch facts of kernel `which` (0 step, 1 calc_p2, 2 linearize) for this system. */
int  trepb_kernel_info(trepb_system* sys, int which, int32_t* regs, int32_t* local_bytes,
                       int32_t* blocks_per_sm, int32_t* block, int32_t* smem_bytes);
/* Host-only (no device needed): check a description; emit the generated constexpr-system type
 * `struct_name` for it (returns required size incl. NUL, writes at most `cap` bytes; -1 on an
 * invalid description); structural hash used to match specialised kernels. */
int  trepb_validate(const trepb_sysdesc* desc);
int  trepb_codegen(const trepb_sysdesc* desc, const char* struct_name, char* buf, int cap);
/* The same with every number of this one description as a literal (no run-time parameters; matched by
 * trepb_desc_hash): a few percent faster, built for the systems BASELINE.json's configs name exactly. */
int  trepb_codegen_literal(const trepb_sysdesc* desc, const char* struct_name, char* buf, int cap);
uint64_t trepb_desc_hash(const trepb_sysdesc* desc);     /* the whole description, parameters included */
/* Hash of the STRUCTURE only: sizes, topology, plugin kinds and index arguments, and which numeric entries are
 * exactly zero.  Specialised kernels are compiled per structure; masses, inertias, lengths, gravity, spring /
 * damping constants, tolerances and spline tables are run-time parameters handed to the kernel as an argument
 * block, so e.g. a damped pendulum with any mass and length runs the kernel built for examples/damped-pendulum.py. */
uint64_t trepb_struct_hash(const trepb_sysdesc* desc);
/* Host-only: the shape the cooperative kernels see for this system, out[10] = nd, nk, nu, nc,
 * links (variable frames), constraint end points, chain pairs, link-tree levels, dynamic configs
 * and configs that some constraint depends on.  A cooperative
 * kernel instantiated for these sizes serves every system of that shape (the link tables stay
 * run-time data).  TREPB_ERR_UNSUPPORTED when the cooperative kernels do not apply. */
int  trepb_coop_dims(const trepb_sysdesc* desc, int32_t* out);
int  trepb_num_specialized(void);
const char* trepb_specialized_name(int i);

/* Per-batch arguments of a step.  Scalars apply to every instance. */
typedef struct trepb_step_args {
    int64_t batch;       /* B                                                              */
    int32_t nsteps;      /* consecutive steps per instance (>= 1)                          */
    int32_t max_iterations; /* Newton cap; reference default 200 (midpointvi.py:174)       */
    double  t0;          /* time of the incoming state (t1 of the first step)              */
    double  dt;          /* step length                                                    */
    double  tolerance;   /* DEL tolerance; reference default 1e-10 (midpointvi.py:20)      */
    /* inputs */
    const double* q1;    /* [B][nq]  state configuration                                   */
    const double* p1;    /* [B][nd]  state momentum                                        */
    const double* u1;    /* [B][nsteps][nu] or NULL if nu == 0 (or to use zeros)           */
    const double* k2;    /* [B][nsteps][nk] kinematic configs at the end of each step      */
    const double* q2_guess;     /* [B][nd] Newton start for the FIRST step, or NULL (= q1) */
    const double* lambda_guess; /* [B][nc] or NULL (= 0)                                   */
    /* outputs (state after the last step) */
    double* q2;          /* [B][nq]                                                        */
    double* p2;          /* [B][nd]                                                        */
    double* lambda1;     /* [B][nc]  may be NULL when nc == 0                              */
    int32_t* iters;      /* [B] Newton iterations summed over the steps; may be NULL       */
    int32_t* status;     /* [B] 0 ok, -1 not converged, -2 singular Jacobian               */
    /* optional trajectory capture: every `sample_every`-th step's (q2,p2), 0 = off        */
    int32_t sample_every;
    int32_t _pad;
    double* traj_q;      /* [B][nsteps/sample_every][nq] */
    double* traj_p;      /* [B][nsteps/sample_every][nd] */
    /* optional time grid shared by the batch: step s runs from times[s] to times[s+1] (the reference steps
     * on arbitrary self._time[k], trep/discopt/dsystem.py:229-250, 426-457); NULL: t0 + s dt accumulated
     * as t2 = t1 + dt.  Device pointer for the _dev entry point. */
    const double* times; /* [nsteps+1] or NULL */
} trepb_step_args;

/* Host-pointer entry points stage through device buffers owned by the handle.  trepb_step_batch and
 * trepb_linearize_batch cut a batch of >= 2^17 instances into 2 or 4 contiguous chunks that alternate between two
 * streams, so that the host<->device copies of one chunk overlap the kernel of another (pinned host buffers make the
 * copies asynchronous); results are bit-identical to one launch over the whole batch.                       */
int trepb_step_batch(trepb_system* sys, const trepb_step_args* args);                   /* host pointers   */
int trepb_step_batch_dev(trepb_system* sys, const trepb_step_args* args, void* stream); /* device pointers */

/* Closed-loop rollouts with an affine feedback inside the time loop: DSystem.project
 * (trep/discopt/dsystem.py:426-457) and DOptimizer.armijo_simulate (trep/discopt/doptimizer.py:405-428),
 * for a batch of (bX, bU) candidates - e.g. every Armijo step size of one line search at once:
 *     X[0] = bX[0];   U[k] = bU[k] - K[k] (X[k] - bX[k]);   X[k+1] = f(X[k], U[k], k)
 * in the DSystem layout  X = [Q(nq); p(nd); v(nk)],  U = [u(nu); rho(nk)]  (dsystem.py:19-66);
 * f is one MidpointVI step (set() for k = 0: lambda starts from 0; step() afterwards: lambda carried). */
typedef struct trepb_project_args {
    int64_t batch;          /* B candidates                                                     */
    int32_t nsteps;         /* K steps; bX / X hold K+1 states                                  */
    int32_t max_iterations;
    double  t0, dt, tolerance;
    const double* bX;       /* [B][K+1][nX]                                                     */
    const double* bU;       /* [B][K][nU]                                                       */
    const double* Kfb;      /* [K][nU][nX] shared by the batch, or [B][K][nU][nX]               */
    int32_t k_per_instance; /* 0: Kfb shared, 1: one gain sequence per candidate                */
    int32_t use_hint;       /* 1: Newton start of step k = dynamic configs of bX[k+1] (project's
                               xk_hint); 0: = current configuration (armijo_simulate)           */
    double* X;              /* [B][K+1][nX] out                                                 */
    double* U;              /* [B][K][nU]   out                                                 */
    int32_t* iters;         /* [B] Newton iterations summed over the steps; may be NULL         */
    int32_t* status;        /* [B] 0 ok, -1 not converged, -2 singular                          */
    int32_t* fail_step;     /* [B] first failed step (K if none): armijo_simulate returns the
                               partial trajectory X[:k], U[:k]; may be NULL                     */
    const double* times;    /* [K+1] time grid shared by the batch (DSystem.time), or NULL: t0 + k dt */
} trepb_project_args;

int trepb_project_batch(trepb_system* sys, const trepb_project_args* args);
int trepb_project_batch_dev(trepb_system* sys, const trepb_project_args* args, void* stream);

/* Time-varying discrete LQR, batched over rollouts: trep.discopt.dlqr.solve_tv_lqr
 * (trep/discopt/dlqr.py:9-38), the Riccati sweep behind DSystem.calc_feedback_controller
 * (trep/discopt/dsystem.py:474-494).  It consumes the A / B slabs trepb_linearize_batch_dev wrote
 * ([rollout][k] order) and produces the gains in the per-candidate layout trepb_project_batch reads,
 * so linearize -> LQR -> project runs without leaving the GPU.  No system handle is needed.
 *     P = Q(K);  for k = K-1..0:  gamma = R(k) + B^T P B,  Kp = B^T P A,  K[k] = gamma^-1 Kp,
 *                                 P = Q(k) + A^T P A - Kp^T K[k],  P = (P + P^T)/2                  */
typedef struct trepb_lqr_args {
    int64_t batch;        /* rollouts                                                   */
    int32_t nsteps;       /* K                                                          */
    int32_t nX, nU;
    int32_t q_per_step;   /* 0: Q is one [nX][nX] matrix, 1: Q is [K+1][nX][nX]         */
    int32_t r_per_step;   /* 0: R is one [nU][nU] matrix, 1: R is [K][nU][nU]           */
    int32_t _pad;
    const double* A;      /* [batch][K][nX][nX]                                         */
    const double* B;      /* [batch][K][nX][nU]                                         */
    const double* Q;
    const double* R;
    double* Kfb;          /* [batch][K][nU][nX] out                                     */
    double* P0;           /* [batch][nX][nX] out (P at k = 0), may be NULL              */
    int32_t* status;      /* [batch] 0 ok, -2 singular gamma                            */
} trepb_lqr_args;

int trepb_lqr_batch(int device, const trepb_lqr_args* args);                   /* host pointers   */
int trepb_lqr_batch_dev(int device, const trepb_lqr_args* args, void* stream); /* device pointers */

/* Time-varying discrete LQ problem with linear and cross cost terms, batched over rollouts:
 * trep.discopt.dlqr.solve_tv_lq (trep/discopt/dlqr.py:41-81), the solve inside
 * DOptimizer.calc_descent_direction (trep/discopt/doptimizer.py:228-318).
 *     P = Q(K), b = q[K];  for k = K-1..0:
 *         gamma = R(k) + B^T P B,  Kp = B^T P A + S(k)^T,  C[k] = gamma^-1 (B^T b + r[k]),  K[k] = gamma^-1 Kp,
 *         b = q[k] - K[k]^T r[k] + (A^T - K[k]^T B^T) b,   P = Q(k) + A^T P A - Kp^T K[k],  P = (P + P^T)/2
 * Same kernel as trepb_lqr_batch (one CTA per rollout, P / P A / A[k] in shared memory); the affine
 * recursion rides along as one more right-hand side of the gamma factorization.               */
typedef struct trepb_lq_args {
    int64_t batch;            /* rollouts                                                          */
    int32_t nsteps;           /* K                                                                 */
    int32_t nX, nU;
    int32_t cost_per_rollout; /* 0: Q, S, R, q, r shared by the batch; 1: one set per rollout      */
    const double* A;          /* [batch][K][nX][nX]                                                */
    const double* B;          /* [batch][K][nX][nU]                                                */
    const double* Q;          /* ([batch])[K+1][nX][nX]                                            */
    const double* S;          /* ([batch])[K][nX][nU] cross term, NULL = zero                      */
    const double* R;          /* ([batch])[K][nU][nU]                                              */
    const double* q;          /* ([batch])[K+1][nX]                                                */
    const double* r;          /* ([batch])[K][nU]                                                  */
    double* Kfb;              /* [batch][K][nU][nX] out                                            */
    double* C;                /* [batch][K][nU] out (affine part of the optimal control)           */
    double* P0;               /* [batch][nX][nX] out, may be NULL                                  */
    double* b0;               /* [batch][nX] out, may be NULL                                      */
    int32_t* status;          /* [batch] 0 ok, -2 singular gamma                                   */
} trepb_lq_args;

int trepb_lq_batch(int device, const trepb_lq_args* args);                   /* host pointers   */
int trepb_lq_batch_dev(int device, const trepb_lq_args* args, void* stream); /* device pointers */
/* Device time of the last Riccati kernel launched on `device` by any of the four calls above (CUDA events on the
 * launching stream; waits for that kernel).  For nX >= 32 every product runs on the FP64 tensor cores
 * (mma.sync m8n8k4, 16 x 40 warp tiles, ragged edges read as zero), below that on 4 x 4 register tiles; the
 * gamma solve is a Gauss-Jordan elimination by the whole CTA (nU (nU + nX + 1) <= 2048).                  */
int trepb_lqr_last_kernel_ms(int device, float* ms);

/* Tangent (forward) sweep about a linearization, batched over rollouts: DSystem.dproject
 * (trep/discopt/dsystem.py:460-471) and the last loop of DOptimizer.calc_descent_direction
 * (trep/discopt/doptimizer.py:348-402):
 *     dX[0] = x0 (NULL: bdX[0], or zero when bdX is NULL);
 *     dU[k] = bdU[k] - K[k] (dX[k] - bdX[k]);   dX[k+1] = A[k] dX[k] + B[k] dU[k]
 * It reads the A / B slabs trepb_linearize_batch_dev writes and the gains of trepb_lqr_batch_dev /
 * trepb_lq_batch_dev as they are.  No system handle is needed.  One team of lanes per rollout streams
 * each step through shared memory; every output element is summed in a fixed order, so a rollout gives
 * the same bits alone and inside any batch.  nU = 0 is allowed (B, K, bdU and dU may then be NULL).  */
typedef struct trepb_tangent_args {
    int64_t batch;            /* rollouts                                              */
    int32_t nsteps;           /* K                                                     */
    int32_t nX, nU;
    int32_t _pad;
    const double* A;          /* [batch][K][nX][nX]                                    */
    const double* B;          /* [batch][K][nX][nU]                                    */
    const double* K;          /* [batch][K][nU][nX]                                    */
    const double* bdX;        /* [batch][K+1][nX], NULL = zero                         */
    const double* bdU;        /* [batch][K][nU], NULL = zero                           */
    const double* x0;         /* [batch][nX] dX[0], NULL = bdX[0] (zero without bdX)   */
    double* dX;               /* [batch][K+1][nX] out                                  */
    double* dU;               /* [batch][K][nU] out                                    */
} trepb_tangent_args;

int trepb_tangent_batch(int device, const trepb_tangent_args* args);                   /* host pointers   */
int trepb_tangent_batch_dev(int device, const trepb_tangent_args* args, void* stream); /* device pointers */

/* Adjoint (backward) sweep, batched over rollouts: the costate recursion of DOptimizer.calc_newton_model
 * (trep/discopt/doptimizer.py:319-345),
 *     z[K] = m_dx;   z[k] = l_dx[k] - K[k]^T l_du[k] + A[k]^T z[k+1] - K[k]^T (B[k]^T z[k+1]),
 * evaluated as l_dx[k] + A[k]^T z[k+1] - K[k]^T (l_du[k] + B[k]^T z[k+1]) (A - B K is never formed).
 * K NULL gives the open-loop costate z[k] = l_dx[k] + A[k]^T z[k+1].  Same layouts and team scheme as
 * trepb_tangent_batch.  z1, if given, receives z[k+1] for k < K, packed [batch][K][nX]: the costate each step's
 * z-contracted second derivatives take (trepb_deriv2_batch_dev's z over the batch x K step instances).  */
typedef struct trepb_adjoint_args {
    int64_t batch;            /* rollouts                                              */
    int32_t nsteps;           /* K                                                     */
    int32_t nX, nU;
    int32_t _pad;
    const double* A;          /* [batch][K][nX][nX]                                    */
    const double* B;          /* [batch][K][nX][nU], needed with K                     */
    const double* K;          /* [batch][K][nU][nX], NULL = open loop                  */
    const double* l_dx;       /* [batch][K][nX], NULL = zero                           */
    const double* l_du;       /* [batch][K][nU], NULL = zero                           */
    const double* m_dx;       /* [batch][nX]                                           */
    double* z;                /* [batch][K+1][nX] out                                  */
    double* z1;               /* [batch][K][nX] out (z[k+1]), may be NULL              */
} trepb_adjoint_args;

int trepb_adjoint_batch(int device, const trepb_adjoint_args* args);                   /* host pointers   */
int trepb_adjoint_batch_dev(int device, const trepb_adjoint_args* args, void* stream); /* device pointers */

/* Quadratic tracking cost and its LQ model, batched over trajectories: trep.discopt.DCost (dcost.py) as
 * DOptimizer.calc_cost / calc_dcost sum it (doptimizer.py).  With dx_k = X[k] - Xd[k], du_k = U[k] - Ud[k]:
 *     cost  = sum_{k<K} (dx_k^T Q dx_k + du_k^T R du_k) / 2 + dx_K^T Q dx_K / 2
 *     q[k]  = dx_k^T Q (k = 0..K),   r[k] = du_k^T R
 *     dcost = sum_{k<K} (q[k] . dX[k] + r[k] . dU[k]) + q[K] . dX[K]
 *     Qm[k] = Q (+ fdxdx[k] for k < K),   Sm[k] = 0 (+ fdxdu[k]),   Rm[k] = R (+ fdudu[k])
 * Trajectory b tracks reference ref_index[b] (NULL: every trajectory tracks reference 0).  Every output is
 * optional; q, r, Qm, Sm and Rm are in the per-rollout layout trepb_lq_batch_dev reads (cost_per_rollout = 1),
 * l_dx / m_dx in the layout trepb_adjoint_batch_dev reads, and the three Newton blocks in the layout
 * trepb_deriv2_batch_dev writes over the batch x K step instances.  Every sum runs in ascending index order with
 * separately rounded products and additions, so a trajectory gives the same bits alone and inside any batch, and
 * each Newton sum is one IEEE addition.  No system handle is needed.  nU = 0 is allowed.                     */
typedef struct trepb_track_args {
    int64_t batch;            /* trajectories                                          */
    int32_t nsteps;           /* K                                                     */
    int32_t nX, nU;
    int32_t nref;             /* references in Xd / Ud (>= 1)                          */
    const double* X;          /* [batch][K+1][nX]                                      */
    const double* U;          /* [batch][K][nU]                                        */
    const double* Xd;         /* [nref][K+1][nX]                                       */
    const double* Ud;         /* [nref][K][nU]                                         */
    const double* Q;          /* [nX][nX]                                              */
    const double* R;          /* [nU][nU]                                              */
    const int32_t* ref_index; /* [batch], NULL = reference 0 for all                   */
    const double* dX;         /* [batch][K+1][nX], needed with dcost                   */
    const double* dU;         /* [batch][K][nU], needed with dcost                     */
    const double* fdxdx;      /* [batch*K][nX][nX] Newton blocks: all three or none    */
    const double* fdxdu;      /* [batch*K][nX][nU]                                     */
    const double* fdudu;      /* [batch*K][nU][nU]                                     */
    double* cost;             /* [batch] out                                           */
    double* dcost;            /* [batch] out                                           */
    double* q;                /* [batch][K+1][nX] out                                  */
    double* r;                /* [batch][K][nU] out                                    */
    double* l_dx;             /* [batch][K][nX] out (q[:K])                            */
    double* m_dx;             /* [batch][nX] out (q[K])                                */
    double* Qm;               /* [batch][K+1][nX][nX] out                              */
    double* Sm;               /* [batch][K][nX][nU] out                                */
    double* Rm;               /* [batch][K][nU][nU] out                                */
} trepb_track_args;

int trepb_track_batch(int device, const trepb_track_args* args);                   /* host pointers   */
int trepb_track_batch_dev(int device, const trepb_track_args* args, void* stream); /* device pointers */

/* Armijo line-search candidates of DOptimizer.armijo_search (doptimizer.py), ncand step sizes for each of `groups`
 * rollouts at once: for group g (rollout rows[g], NULL = g) and step size lam[m],
 *     bX[g][m] = X + lam[m] dX,   bU[g][m] = U + lam[m] dU   (product and sum rounded separately)
 *     Kc[g][m] = Kproj                                        (per-candidate gains for trepb_project_batch_dev
 *                                                              with k_per_instance = 1)                         */
typedef struct trepb_candidates_args {
    int64_t groups;           /* rollouts searched                                     */
    int32_t ncand;            /* M step sizes per rollout (>= 1)                       */
    int32_t nsteps;           /* K                                                     */
    int32_t nX, nU;
    int64_t nrollouts;        /* rollouts in X .. Kproj (host form with rows only)     */
    const int32_t* rows;      /* [groups], NULL = identity                             */
    const double* lam;        /* [ncand]                                               */
    const double* X;          /* [R][K+1][nX]                                          */
    const double* U;          /* [R][K][nU]                                            */
    const double* dX;         /* [R][K+1][nX]                                          */
    const double* dU;         /* [R][K][nU]                                            */
    const double* Kproj;      /* [R][K][nU][nX]                                        */
    double* bX;               /* [groups][ncand][K+1][nX] out                          */
    double* bU;               /* [groups][ncand][K][nU] out                            */
    double* Kc;               /* [groups][ncand][K][nU][nX] out                        */
} trepb_candidates_args;

int trepb_candidates_batch(int device, const trepb_candidates_args* args);                   /* host pointers   */
int trepb_candidates_batch_dev(int device, const trepb_candidates_args* args, void* stream); /* device pointers */

/* Stationary discrete LQR, batched over models: the stabilizing solution P of the discrete algebraic Riccati equation
 *     P = A^T P A - (A^T P B + S)(R + B^T P B)^-1 (B^T P A + S^T) + Q
 * and the gain K = (R + B^T P B)^-1 (B^T P A + S^T) (u = -K x), what scipy.linalg.solve_discrete_are (with s = S) and
 * one more solve give on the host.  No counterpart in the reference (discopt.dlqr is time-varying only).  A / B are in
 * the layout trepb_linearize_batch_dev writes for `batch` single-step instances; K [batch][nU][nX] is the layout
 * trepb_project_batch reads with k_per_instance = 1 for a one-step rollout (for K steps, repeat each model's gain K
 * times).  Structure-preserving doubling (quadratic convergence, A need not be invertible), one CTA per model with
 * every matrix in shared memory: 8 (4 n ((n + 1) | 1) + ...) bytes, so nX = 80 runs with any nU <= 39 and nX <= 82
 * with nU = 1; larger shapes are TREPB_ERR_UNSUPPORTED.  Every output element is summed by one thread in a fixed
 * order, so a model gives the same bits alone and inside any batch; P is symmetric bit for bit.  Q is read as
 * (Q + Q^T) / 2.  The K / P rows of a model whose status is not TREPB_DARE_OK are unspecified.  No system handle is
 * needed. */
#define TREPB_DARE_OK 0
#define TREPB_DARE_NOT_CONVERGED -1 /* ||H' - H||_F > tol ||H'||_F after max_iterations doublings, or the
                                       doubling stalled on a P whose residual exceeds 1e-6 of the equation's terms */
#define TREPB_DARE_SINGULAR -2      /* exact zero pivot in R, in I + G H or in R + B^T P B (the LQR kernel's code) */
#define TREPB_DARE_NONFINITE -3     /* an iterate overflowed or went NaN (e.g. an unstable mode B cannot reach)   */
typedef struct trepb_dare_args {
    int64_t batch;            /* models                                                              */
    int32_t nX, nU;
    int32_t max_iterations;   /* doubling steps (64 is ample: the error squares every step)          */
    int32_t q_per_rollout;    /* 0: Q is one [nX][nX] matrix, 1: [batch][nX][nX]                     */
    int32_t r_per_rollout;    /* 0: R is one [nU][nU] matrix, 1: [batch][nU][nU]                     */
    int32_t s_per_rollout;    /* 0: S is one [nX][nU] matrix, 1: [batch][nX][nU]                     */
    double tol;               /* stop at ||H' - H||_F <= tol ||H'||_F (1e-13 is about 60 ulp)         */
    const double* A;          /* [batch][nX][nX]                                                     */
    const double* B;          /* [batch][nX][nU]                                                     */
    const double* Q;
    const double* R;
    const double* S;          /* cross term, NULL = zero                                             */
    double* K;                /* [batch][nU][nX] out, may be NULL                                    */
    double* P;                /* [batch][nX][nX] out, may be NULL                                    */
    int32_t* status;          /* [batch] TREPB_DARE_*                                                 */
    int32_t* iterations;      /* [batch] doubling steps taken, may be NULL                           */
} trepb_dare_args;

int trepb_dare_batch(int device, const trepb_dare_args* args);                   /* host pointers   */
int trepb_dare_batch_dev(int device, const trepb_dare_args* args, void* stream); /* device pointers */

/* Closed-loop cost and stability of stationary gains, batched over (gain, model) pairs: the solution P of the discrete
 * Lyapunov (Stein) equation
 *     P = A_c^T P A_c + Q_c,   A_c = A - B K,   Q_c = Q - S K - K^T S^T + K^T R K
 * for gain K under model (A, B), the infinite-horizon cost-to-go of u = -K x under the stage cost
 * x^T Q x + 2 x^T S u + u^T R u, which exists exactly when rho(A_c) < 1: what scipy.linalg.solve_discrete_lyapunov
 * (A_c^T, Q_c) gives on the host, with a stability verdict.  No counterpart in the reference.  Pair p evaluates gain
 * gain_index[p] under model model_index[p] (either NULL: gain p / model p), so a G x M cross-evaluation of the gains
 * trepb_dare_batch wrote under the models trepb_linearize_batch_dev wrote is one call.  Smith doubling
 * (P <- P + F^T P F, F <- F F from P = Q_c, F = A_c) until ||dP||_F <= tol ||P||_F and ||F||_F <= tol, one CTA per
 * pair with A_c, P, F and one work block in shared memory: 8 (4 n ((n + 1) | 1) + ...) bytes; every shape
 * trepb_dare_batch admits is admitted (up to nX = 84 at nU = 1 on a 227 KB device), larger ones are
 * TREPB_ERR_UNSUPPORTED.  Every output element is summed by one thread in a fixed order, so a pair gives the same bits
 * alone and inside any batch; P is symmetric bit for bit.  Q and R are read as (Q + Q^T) / 2 and (R + R^T) / 2.  The
 * P rows of a pair whose status is not TREPB_DLYAP_STABLE are unspecified and its cost is +inf.  The host entry
 * refuses an index outside [0, gains) / [0, models); the _dev entry cannot read the indices before the launch and
 * reports such a pair as TREPB_DLYAP_BAD_INDEX instead.  No system handle is needed. */
#define TREPB_DLYAP_STABLE 0
#define TREPB_DLYAP_NOT_CONVERGED -1 /* bounded but not shrinking F (rho(A_c) >= 1, e.g. on the unit circle), too slow
                                        to converge within max_iterations, or a residual above 1e-6 of the terms */
#define TREPB_DLYAP_NONFINITE -3     /* an iterate overflowed or went NaN (rho(A_c) > 1 usually ends here)        */
#define TREPB_DLYAP_BAD_INDEX -4     /* _dev entry only: gain_index / model_index outside [0, gains) / [0, models)  */
typedef struct trepb_dlyap_args {
    int64_t pairs;            /* (gain, model) pairs evaluated                                        */
    int64_t gains;            /* G: gains in K (>= pairs without gain_index)                          */
    int64_t models;           /* M: models in A / B (>= pairs without model_index)                    */
    int32_t nX, nU;
    int32_t max_iterations;   /* doubling steps (64 is ample: F squares every step)                    */
    int32_t q_per_model;      /* 0: Q is one [nX][nX] matrix, 1: [models][nX][nX]                     */
    int32_t r_per_model;      /* 0: R is one [nU][nU] matrix, 1: [models][nU][nU]                     */
    int32_t s_per_model;      /* 0: S is one [nX][nU] matrix, 1: [models][nX][nU]                     */
    int32_t x0_per_pair;      /* 0: x0 is one [nX] vector, 1: [pairs][nX]                             */
    double tol;               /* stop at ||dP||_F <= tol ||P||_F and ||F||_F <= tol                    */
    const double* A;          /* [models][nX][nX]                                                     */
    const double* B;          /* [models][nX][nU]                                                     */
    const double* K;          /* [gains][nU][nX], u = -K x                                            */
    const double* Q;
    const double* R;
    const double* S;          /* cross term, NULL = zero                                              */
    const int32_t* gain_index;  /* [pairs], NULL = pair p evaluates gain p                             */
    const int32_t* model_index; /* [pairs], NULL = pair p runs under model p                           */
    const double* x0;         /* cost = x0^T P x0; NULL: see W                                        */
    const double* W;          /* [nX][nX], cost = trace(P W) (x0 and W exclusive, one needed for cost) */
    double* P;                /* [pairs][nX][nX] out, may be NULL                                     */
    double* cost;             /* [pairs] out, may be NULL                                             */
    int32_t* status;          /* [pairs] TREPB_DLYAP_*                                                 */
    int32_t* iterations;      /* [pairs] doubling steps taken, may be NULL                            */
} trepb_dlyap_args;

int trepb_dlyap_batch(int device, const trepb_dlyap_args* args);                   /* host pointers   */
int trepb_dlyap_batch_dev(int device, const trepb_dlyap_args* args, void* stream); /* device pointers */

/* p2 from two consecutive configurations (initialize_from_configs). q0,q1: [B][nq] -> p: [B][nd] */
int trepb_calc_p2_batch(trepb_system* sys, int64_t batch, double dt,
                        const double* q0, const double* q1, double* p);
int trepb_calc_p2_batch_dev(trepb_system* sys, int64_t batch, double dt,
                            const double* q0, const double* q1, double* p, void* stream);

/* Residual of the DEL equation at given (q1, q2, p1, u1, lambda1): _MidpointVI._calc_f == MidpointVI_calc_f
 * (trep/_trep/midpointvi.c:533-575):  f[0:nd] = p1 + D1L2 + fm2 - Dh(q1)^T lambda1,  f[nd:nd+nc] = h(q2).
 * q1, q2: [B][nq]; p1: [B][nd]; u1: [B][nu] or NULL (zeros); lambda1: [B][nc] or NULL (zeros); f: [B][nd+nc]. */
int trepb_calc_f_batch(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1, const double* q2,
                       const double* p1, const double* u1, const double* lambda1, double* f);
int trepb_calc_f_batch_dev(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1, const double* q2,
                           const double* p1, const double* u1, const double* lambda1, double* f, void* stream);
/* Discrete forcing fm2 = (t2 - t1) F(q_mid, dq, u1) on the dynamic configs: _MidpointVI.discrete_fm2
 * (trep/_trep/midpointvi.c:474-478, 2710-2727).  fm2: [B][nd]. */
int trepb_discrete_fm2_batch(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1,
                             const double* q2, const double* u1, double* fm2);
int trepb_discrete_fm2_batch_dev(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1,
                                 const double* q2, const double* u1, double* fm2, void* stream);

/* One linearization per instance: solve the step from (q1,p1,u1,k2[,guess]) then first
 * derivatives.  A: [B][nX][nX], B: [B][nX][nU] with nX = 2*nq, nU = nu+nk (DSystem layout).
 * Raw first-derivative arrays in the reference's storage layout [wrt][out] are optional. */
typedef struct trepb_lin_args {
    int64_t batch;
    int32_t max_iterations;
    /* 0: instance b reads row b of every input array.  L >= 2: the STATE inputs (q1, p1, q2_guess) are
     * trajectories of L rows, [R][L][..] - DSystem's X, or the trajectory capture of trepb_step_batch - and
     * instance b = r (L-1) + k linearizes step k -> k+1 of trajectory r: it reads state row r L + k (pass
     * q2_guess = q1 + nq to use X[k+1] as the Newton start, DSystem.linearize_trajectory's xk_hint).  The
     * per-STEP inputs (u1, k2, t1, t2, lambda_guess) and every output are packed [R][L-1] (row b), the shape
     * of DSystem's U and of linearize_trajectory's A[k], B[k] (trep/discopt/dsystem.py:406-423).  The junk
     * instance that would pair the last state of one trajectory with the first of the next does not exist. */
    int32_t traj_len;
    double  tolerance;
    const double* t1;    /* [B] or NULL -> use t1_scalar */
    const double* t2;    /* [B] or NULL -> use t1_scalar + dt_scalar */
    double  t1_scalar, dt_scalar;
    const double* q1; const double* p1; const double* u1; const double* k2;  /* [B][nq],[B][nd],[B][nu],[B][nk] */
    const double* q2_guess; const double* lambda_guess;                      /* [B][nd],[B][nc] or NULL */
    double* q2; double* p2; double* lambda1;       /* may be NULL */
    int32_t* iters; int32_t* status;               /* iters may be NULL */
    double* A; double* B;                          /* may be NULL */
    double* q2_dq1; double* q2_dp1; double* q2_du1; double* q2_dk2;  /* [B][nq|nd|nu|nk][nd] or NULL */
    double* p2_dq1; double* p2_dp1; double* p2_du1; double* p2_dk2;
    double* l1_dq1; double* l1_dp1; double* l1_du1; double* l1_dk2;  /* [B][..][nc] or NULL */
} trepb_lin_args;

int trepb_linearize_batch(trepb_system* sys, const trepb_lin_args* args);
int trepb_linearize_batch_dev(trepb_system* sys, const trepb_lin_args* args, void* stream);

/* Second derivatives of the discrete flow: _MidpointVI._calc_deriv2 == MidpointVI_calc_deriv2
 * (trep/_trep/midpointvi.c:2516-2545), after the same solve + first derivatives as
 * trepb_linearize_batch (all of `lin`'s outputs stay optional).  Tensors use the reference's
 * storage layout [B][wrt A][wrt B][output] (trep/_trep/trep.h:439-473, getters
 * trep/midpointvi.py:366-731); same-type pairs are stored in full (both symmetric halves).
 *   d2[10*which + kind]   which: 0 q2 (output = nd), 1 p2 (nd), 2 lambda1 (nc)
 *                         kind : 0 q1q1  1 q1p1  2 q1u1  3 q1k2  4 p1p1  5 p1u1  6 p1k2
 *                                7 u1u1  8 u1k2  9 k2k2          (q1: nq, p1: nd, u1: nu, k2: nk)
 * Any entry may be NULL. */
typedef struct trepb_d2_args {
    trepb_lin_args lin;
    double* d2[30];
    /* Optional z-contracted forms, what DSystem.fdxdx(z) / fdxdu(z) / fdudu(z) return
     * (trep/discopt/dsystem.py:320-386): sum over outputs of z_Qd * q2_dAdB + z_p * p2_dAdB,
     * assembled in the DSystem state/input layout.  z: [B][nX] (only its Qd and p parts are read);
     * fdxdx: [B][nX][nX], fdxdu: [B][nX][nU], fdudu: [B][nU][nU]; all NULL to skip.  This is the
     * form the optimizer consumes (65 KB instead of 1.76 MB per marionette instance). */
    const double* z;
    double* fdxdx;
    double* fdxdu;
    double* fdudu;
} trepb_d2_args;

int trepb_deriv2_batch(trepb_system* sys, const trepb_d2_args* args);
int trepb_deriv2_batch_dev(trepb_system* sys, const trepb_d2_args* args, void* stream);

/* ---- per-instance physical parameters ------------------------------------------------------
 * The entry points above run every instance of a batch on the numbers of the one description behind the handle.
 * The *_varied_batch* entry points take the same arguments plus a trepb_varied: n entries of the description's
 * numeric tables, and one row of n values per instance, which override those entries for that instance (every
 * other entry keeps the description's value): Monte Carlo over uncertain masses / lengths / gains, one candidate
 * parameter set per instance in system identification, K plausible models in robust trajectory optimisation.
 *   rows       one per instance; trepb_linearize_varied_batch* with traj_len >= 2: one per trajectory r (all
 *              traj_len - 1 steps of a rollout share its physics).  trepb_deriv2_varied_batch* takes one row per
 *              instance only: args->lin.traj_len must be 0 (TREPB_ERR_INVALID otherwise).
 *   entries    only run-time parameters can vary: an entry whose description value is exactly 0, or +-1 in
 *              frame_se3, is structure (it folds away in the specialised kernels and in trepb_struct_hash), and
 *              so are the spline x-points of a NonlinearConfigSpring and a Gravity component whose sum over all
 *              Gravity potentials is 0.  Such an entry, an index out of range or an entry named twice is
 *              TREPB_ERR_INVALID (trepb_last_error names it).  A varied Gravity component re-forms the
 *              gravity sum per instance.  A row value of exactly 0 is not checked and keeps the entry's role.
 *   kernels    specialised and table-driven thread kernels (a handle built for an all-literal instantiation runs
 *              the run-time-parameter kernels of its structure).  Cooperative handles run the varied cooperative
 *              kernels of their flavour when created with TREPB_FLAG_COOP_VARIED (each team re-evaluates its own
 *              copy of the link tables from its row) and are TREPB_ERR_UNSUPPORTED without it (or create the handle
 *              with TREPB_FLAG_NO_COOP for the thread kernels).  Second derivatives vary through the same kernels
 *              and schemes as the plain call (the per-pair kernel, or the per-parameter scheme on the tables);
 *              its linearize launch runs on the same rows (on a flagged cooperative handle: the varied cooperative
 *              linearize kernel).
 * Results equal those of a handle created from each instance's own description, run through the plain entry
 * point, bit for bit - with one exception on cooperative handles: a varied angle of a constant rotation frame
 * (TREPB_PAR_FRAME_VALUE of an RX / RY / RZ frame without a config) takes its cos / sin from the device math
 * library, a handle built on the host from the C library; they may differ in the last bit, and the results
 * then agree to the project's parity tolerance, not bit for bit. */
#define TREPB_PAR_FRAME_VALUE 0   /* index f           */
#define TREPB_PAR_FRAME_SE3 1     /* index 12 f + k    */
#define TREPB_PAR_FRAME_MASS 2    /* index 4 f + k     */
#define TREPB_PAR_POT_D 3         /* index 4 i + k     */
#define TREPB_PAR_FORCE_D 4       /* index 4 i + k     */
#define TREPB_PAR_CON_D 5         /* index 4 i + k     */
#define TREPB_PAR_DPOOL 6         /* index k           */
typedef struct trepb_varied {
    int32_t n, _pad;          /* number of varied entries                                                   */
    const int32_t* table;     /* [n] TREPB_PAR_* (host pointer)                                             */
    const int32_t* index;     /* [n] flat index into that table (host pointer)                              */
    const double*  values;    /* [rows][n]: row r = that instance's (trajectory's) values; device pointer for
                                 the _dev entry points, host pointer otherwise                               */
} trepb_varied;
/* Host-only: checks a trepb_varied's entries against a description (values are not read). */
int trepb_varied_check(const trepb_sysdesc* desc, const trepb_varied* v);
int trepb_step_varied_batch(trepb_system* sys, const trepb_step_args* args, const trepb_varied* v);
int trepb_step_varied_batch_dev(trepb_system* sys, const trepb_step_args* args, const trepb_varied* v, void* stream);
int trepb_linearize_varied_batch(trepb_system* sys, const trepb_lin_args* args, const trepb_varied* v);
int trepb_linearize_varied_batch_dev(trepb_system* sys, const trepb_lin_args* args, const trepb_varied* v, void* stream);
int trepb_project_varied_batch(trepb_system* sys, const trepb_project_args* args, const trepb_varied* v);
int trepb_project_varied_batch_dev(trepb_system* sys, const trepb_project_args* args, const trepb_varied* v, void* stream);
int trepb_calc_p2_varied_batch(trepb_system* sys, int64_t batch, double dt, const double* q0, const double* q1,
                               double* p, const trepb_varied* v);
int trepb_calc_p2_varied_batch_dev(trepb_system* sys, int64_t batch, double dt, const double* q0, const double* q1,
                                   double* p, const trepb_varied* v, void* stream);
int trepb_calc_f_varied_batch(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1,
                              const double* q2, const double* p1, const double* u1, const double* lambda1, double* f,
                              const trepb_varied* v);
int trepb_calc_f_varied_batch_dev(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1,
                                  const double* q2, const double* p1, const double* u1, const double* lambda1,
                                  double* f, const trepb_varied* v, void* stream);
int trepb_discrete_fm2_varied_batch(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1,
                                    const double* q2, const double* u1, double* fm2, const trepb_varied* v);
int trepb_discrete_fm2_varied_batch_dev(trepb_system* sys, int64_t batch, double t1, double t2, const double* q1,
                                        const double* q2, const double* u1, double* fm2, const trepb_varied* v,
                                        void* stream);
int trepb_deriv2_varied_batch(trepb_system* sys, const trepb_d2_args* args, const trepb_varied* v);
int trepb_deriv2_varied_batch_dev(trepb_system* sys, const trepb_d2_args* args, const trepb_varied* v, void* stream);

/* ---- multi-GPU: one process per GPU ---------------------------------------------------------
 * Instances are independent, so a batch shards over ranks with no exchange during compute (each
 * rank calls the entry points above on its own contiguous block).  The one exchange of the path is
 * collecting the A / B slabs of DSystem.linearize_trajectory (trep/discopt/dsystem.py:406-423) where
 * the sequential Riccati sweep runs (trep/discopt/dlqr.py:9-81).  Device to device over NVLink, two ways:
 *   (1) NCCL on slabs already in local HBM: trepb_comm_allgather_dev (ncclAllGather) or
 *       trepb_comm_gather_dev (grouped ncclSend / ncclRecv to `root`).  NCCL is loaded at run time
 *       (libnccl.so.2: the copy already in the process, else the system one; TREPB_NCCL_LIB overrides).
 *   (2) fused into the linearize kernel: the root exports its slab (trepb_ipc_export), every rank maps
 *       it (trepb_ipc_open) and passes mapped + rank offset as the A / B pointers of
 *       trepb_linearize_batch_dev: the kernel's own stores land in the root's HBM, no second pass.
 * The 128-byte id of trepb_comm_unique_id (rank 0) and the 64-byte IPC handles travel between the
 * processes by the host's own means (trep_b200/dist.py: a TCP rendezvous on MASTER_ADDR/MASTER_PORT). */
#define TREPB_COMM_ID_BYTES 128
#define TREPB_IPC_HANDLE_BYTES 64
typedef struct trepb_comm trepb_comm; /* opaque */
int  trepb_comm_available(int* nccl_version);            /* 0 if NCCL could be loaded */
int  trepb_comm_unique_id(char* id);                     /* id[TREPB_COMM_ID_BYTES], call on one rank */
int  trepb_comm_create(int device, int rank, int nranks, const char* id, trepb_comm** out);  /* collective */
void trepb_comm_destroy(trepb_comm* comm);
int  trepb_comm_rank(const trepb_comm* comm, int* rank, int* nranks);
/* recv: [nranks][bytes_per_rank] on every rank (allgather) / on `root` (gather; may be NULL elsewhere);
 * device pointers, enqueued on `stream`, no synchronization. */
int  trepb_comm_allgather_dev(trepb_comm* comm, const void* send, void* recv, int64_t bytes_per_rank, void* stream);
int  trepb_comm_gather_dev(trepb_comm* comm, const void* send, void* recv, int64_t bytes_per_rank, int root, void* stream);
/* ptr: the BASE of an allocation made by trepb_malloc (cudaMalloc); handle[TREPB_IPC_HANDLE_BYTES]. */
int  trepb_ipc_export(int device, const void* ptr, char* handle);
int  trepb_ipc_open(int device, const char* handle, void** ptr);    /* in ANOTHER process than the exporter */
int  trepb_ipc_close(int device, void* ptr);
/* CUDA-event timing for hosts without a CUDA binding of their own: record(pair, 0 | 1, stream), then
 * elapsed_ms synchronizes on the second event. */
int  trepb_event_pair_create(int device, void** pair);
int  trepb_event_record(void* pair, int which, void* stream);
int  trepb_event_elapsed_ms(void* pair, float* ms);
void trepb_event_pair_destroy(void* pair);

/* Device utilities so that a C host (no torch) can own HBM buffers. */
int trepb_device_count(int* n);
int trepb_malloc(int device, int64_t bytes, void** ptr);
int trepb_free(int device, void* ptr);
int trepb_host_alloc(int64_t bytes, void** ptr);   /* pinned host memory */
int trepb_host_free(void* ptr);
int trepb_memset(int device, void* dst, int value, int64_t bytes);
int trepb_memcpy_h2d(int device, void* dst, const void* src, int64_t bytes);
int trepb_memcpy_d2h(int device, void* dst, const void* src, int64_t bytes);
int trepb_memcpy_d2d(int device, void* dst, const void* src, int64_t bytes);   /* also peer-mapped addresses */
int trepb_synchronize(int device);
/* Time of the most recent kernel launched by a *_dev / host entry point on this system, in
 * milliseconds, measured with CUDA events on the launching stream (valid after a sync). */
int trepb_last_kernel_ms(trepb_system* sys, float* ms);
/* FP64 FMA micro-benchmark (roofline denominator): achieved TFLOP/s of a DFMA-saturating kernel. */
int trepb_measure_fp64_peak(int device, double* tflops);
/* Diagnostic: sin and cos as the kernels compute them (trep/_trep/frame.c:839-1076 calls libm's sin / cos for
 * every revolute frame; the kernels use their own routine with the coefficients in constant memory).  Host
 * pointers, n values.  Used by the tests to bound its error in ulps against libm. */
int trepb_sincos_batch(int device, int64_t n, const double* x, double* s, double* c);

#ifdef __cplusplus
}
#endif
#endif /* TREPB_H */
