/* cmpc.h - C ABI of the B200-native batched convex-MPC solver.
 *
 * Drop-in boundary for the hot path of the reference's `MPC` class
 * (Emilianogith/MPC-for-dynamic-locomotion-in-the-MIT-cheetah-3, src/mpc.py).  The
 * reference has no FFI layer of its own: `MPC.__init__` builds the QP with CasADi
 * (src/mpc.py:49-173) and `MPC.solve` re-parameterises and solves it with OSQP every
 * tick (src/mpc.py:242-258).  Each entry point below names the reference code it
 * replaces.  Python binds these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - All array arguments of the non-`_host` functions are CUDA DEVICE pointers
 *    (e.g. torch `tensor.data_ptr()`), fp32, row-major, contiguous, owned by the caller.
 *  - B problems per call, horizon N fixed per handle (any 1 <= N <= cmpc_max_horizon(), as the
 *    reference accepts any params['N'], src/main.py:41; a horizon without its own compiled kernel
 *    runs on the next compiled one with all-swing, zero-cost padding stages - same optimum).
 *    Legs are FL, FR, HL, HR.
 *      x0     [B,13]      Theta(3) p(3) omega(3) v(3) g        (src/mpc.py:190-198)
 *      r      [B,N,4,3]   lever arms foot - com per stage/leg    (src/mpc.py:218-239)
 *      mask   [B,N] uint8 bit l = 1  <=> leg l in stance at stage i
 *                         (= 1 - swing_param, src/mpc.py:249-254)
 *      x_des  [B,N+1,13]  desired trajectory                     (src/mpc.py:202-214)
 *      mu     [B]         friction coefficient                   (src/mpc.py:33)
 *      U      [B,N,12]    optimal forces, stage-major (U[:,0,:] is what MPC.solve returns,
 *                         src/mpc.py:267-278); swing legs are exactly 0
 *      X      [B,N+1,13]  predicted states (src/mpc.py:265-266), may be NULL
 *      iters/status [B] int32, pri_res/dua_res [B] fp32; any of them may be NULL
 *  - Work is enqueued on `stream` (a cudaStream_t passed as void*) and is asynchronous.
 *  - Every function returns 0 on success or a negative CMPC_ERR_* code; nothing throws.
 *    `cmpc_last_error()` returns a thread-local description of the last failure.
 *  - A handle owns the warm-start state (previous primal/dual solution per problem slot,
 *    src/mpc.py:270-271) and scratch; one handle must not be used from two threads at once.
 *    Disjoint slot ranges [slot0, slot0+B) of one handle may be in flight on different streams.
 *  - No entry point changes the calling thread's current CUDA device.
 */
#ifndef CMPC_H
#define CMPC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CMPC_VERSION_MAJOR 0
#define CMPC_VERSION_MINOR 3

enum {
  CMPC_OK = 0,
  CMPC_ERR_INVALID = -1,     /* bad argument / unsupported configuration            */
  CMPC_ERR_CUDA = -2,        /* a CUDA runtime call failed (see cmpc_last_error)    */
  CMPC_ERR_UNSUPPORTED = -3, /* horizon or weights outside what the kernels cover   */
  CMPC_ERR_NO_DEVICE = -4    /* no CUDA device: there is NO CPU fallback            */
};

/* per-problem solver status written to `status` */
enum {
  CMPC_STATUS_MAX_ITER = 0,  /* OSQP "maximum iterations reached"                  */
  CMPC_STATUS_SOLVED = 1,
  CMPC_STATUS_NAN = -1       /* non-finite data or iterate                          */
};

/* warm-start policy of cmpc_solve */
enum {
  CMPC_WARM_NONE = 0,   /* x = y = 0 every call                                     */
  CMPC_WARM_PRIMAL = 1, /* reference semantics: previous x unshifted, y = 0
                           (src/mpc.py:270-271; CasADi passes lam_g0 = 0)           */
  CMPC_WARM_PRIMAL_DUAL = 2 /* previous x and y                                     */
};

typedef struct cmpc_config {
  int32_t N;            /* horizon, src/main.py:41 (`params['N']`)                   */
  int32_t max_batch;    /* problem slots with persistent warm-start state            */
  float dt;             /* `world_time_step`, src/mpc.py:31                          */
  float mass;           /* src/mpc.py:71                                             */
  float ibody_inv[3];   /* src/mpc.py:73-76                                          */
  float w[13];          /* state weights, src/mpc.py:121-134                         */
  float r_weight;       /* force weight, src/mpc.py:121 (0.0)                        */
  float f_min, f_max;   /* src/mpc.py:45-46                                          */
  float rho, sigma, alpha;   /* ADMM penalty / prox weight / relaxation              */
  float eps_abs, eps_rel;    /* OSQP-style termination tolerances (defaults 1e-3)    */
  int32_t max_iter;     /* src/mpc.py:51 (1000)                                      */
  int32_t check_every;  /* termination test period                                   */
  int32_t refresh_every;/* exact recomputation period of the wrench-space gradient   */
  int32_t warm_mode;    /* CMPC_WARM_*                                               */
  int32_t adaptive_rho_interval; /* OSQP-style rho adaptation every k iterations, 0 = off */
  float adaptive_rho_tolerance;  /* refactor when rho changes by more than this factor (5) */
  float rho_min, rho_max;        /* clamp of the adapted rho                                 */
  int32_t kernel_variant; /* 0 = default kernel of the horizon; 5 = the other formulation where one is
                             compiled (cmpc_has_variant): the stage-wise (Riccati) kernel for N = 10, 12, 16
                             (default: dense), the dense kernel for N = 20, 30 (default: Riccati).  Any
                             other value runs the default; see DESIGN.md 4 */
  int32_t lpt_schedule; /* >0: batches of at least this size are launched hardest-first
                           (conditioning score), 0 = launch in batch order               */
  int32_t device;       /* CUDA device ordinal                                       */
  int32_t host_zero_copy; /* cmpc_solve_host with page-locked caller buffers: 1 = the solve kernel
                           reads the inputs and writes the results directly in host memory over
                           PCIe (no staging copies, transfers overlap the solve CTA by CTA);
                           0 = chunked cudaMemcpyAsync pipeline                              */
  int32_t cache_factorization; /* 1 = keep every slot's factorisation on the device and reuse it in the
                           next cmpc_solve of that slot while its lever arms (to cache_tol_r), yaw
                           (cache_tol_yaw), contact masks and rho are unchanged - standing robots,
                           static contact schedules (closed-loop use); 0 = refactorise every call.
                           (One entry per gait phase was tried for steady-state walking: the lever
                           arms of successive gait cycles differ by more than a safe tolerance.)
                           Costs 4*6N*(6N+20) bytes per slot.  Compiled for the N = 10 and N = 30 kernels
                           (default thread layout; kernel_variant is ignored; horizons padded onto them
                           included), other horizons: UNSUPPORTED.  Needs check_every to be a multiple of
                           refresh_every (the stopping test then runs on a recomputed gradient).      */
  float cache_tol_r, cache_tol_yaw; /* metres / radians (defaults 2e-3, 2e-3)               */
  int32_t cache_max_iter;  /* a solve that needs more iterations drops its cache entry (30) */
  int32_t time_kernel;  /* 1 = bracket every solve-kernel launch of cmpc_solve with CUDA events on the
                           launching stream (read back with cmpc_last_kernel_ms); 0 = off (default) */
} cmpc_config;

typedef struct cmpc_handle cmpc_handle;

/* Fill `cfg` with the reference's constants (src/mpc.py:45-46,71-76,121-134; src/main.py:31-46)
 * for horizon N and the solver defaults of this library. */
int cmpc_default_config(cmpc_config* cfg, int32_t N, int32_t max_batch);

/* Replaces MPC.__init__ (src/mpc.py:25-173): validates the configuration, precomputes the
 * horizon Gram matrices, allocates warm-start state on cfg->device. */
int cmpc_create(const cmpc_config* cfg, cmpc_handle** out);
int cmpc_destroy(cmpc_handle* h);

/* Replaces `self.opt.set_value(...)` x7 + `self.opt.solve()` + `sol.value(...)`
 * (src/mpc.py:242-271) for B independent problems occupying warm-start slots
 * [slot0, slot0+B).  Device pointers. */
int cmpc_solve(cmpc_handle* h, int32_t B, int32_t slot0,
               const float* x0, const float* r, const uint8_t* mask, const float* x_des,
               const float* mu, float* U, float* X, int32_t* iters, float* pri_res,
               float* dua_res, int32_t* status, void* stream);

/* Same call with HOST pointers; returns when the outputs are in host memory.  Page-locked
 * (cudaHostAlloc / torch pin_memory) buffers are accessed by the kernel in place when
 * cfg.host_zero_copy is set; otherwise, and for pageable buffers, the batch is staged through
 * pinned arenas in two chunks so that H2D / solve / D2H overlap on internal streams.
 * This is the call the reference-facing Python `MPC.solve` drop-in makes. */
int cmpc_solve_host(cmpc_handle* h, int32_t B, int32_t slot0,
                    const float* x0, const float* r, const uint8_t* mask, const float* x_des,
                    const float* mu, float* U, float* X, int32_t* iters, float* pri_res,
                    float* dua_res, int32_t* status);

/* Asynchronous form of cmpc_solve_host for page-locked buffers (cfg.host_zero_copy = 1): the batch is
 * enqueued on the handle's host-path stream and the call returns with a ticket; the buffers belong to the
 * library until cmpc_host_wait(h, ticket) returns.  Submissions are processed in order, so a caller with a
 * stream of batches double-buffers: submit batch k+1, wait for batch k.  The inputs of a submission are copied
 * by the copy engines into one of two device arenas while the previous submission is solved, and its results
 * are copied back while the next one is solved; a ticket completes when the results are in the caller's
 * buffers.  CMPC_ERR_UNSUPPORTED for pageable buffers (use cmpc_solve_host).
 * (No counterpart in the reference, whose solve is synchronous: src/mpc.py:247.) */
int cmpc_solve_host_async(cmpc_handle* h, int32_t B, int32_t slot0,
                          const float* x0, const float* r, const uint8_t* mask, const float* x_des,
                          const float* mu, float* U, float* X, int32_t* iters, float* pri_res,
                          float* dua_res, int32_t* status, int32_t* ticket);
int cmpc_host_wait(cmpc_handle* h, int32_t ticket);

/* Exports the dense condensed QP  min 1/2 u'Hu + g'u  over all 12N forces
 * (H [B,12N,12N], g [B,12N]; rows/columns of swing legs are zero), i.e. what CasADi
 * derives symbolically from src/mpc.py:64-136 after eliminating X.  Problem i uses the body,
 * the cost weights, the external wrench, the force references and the stage weights of slot i
 * (cmpc_set_body, cmpc_set_weights, cmpc_set_wrench, cmpc_set_force_ref, cmpc_set_stage_weights).
 * Device pointers. */
int cmpc_condense(cmpc_handle* h, int32_t B, const float* x0, const float* r,
                  const uint8_t* mask, const float* x_des, float* H, float* g, void* stream);

/* Warm-start state (src/mpc.py:270-271 `set_initial`): forget it (and the cached factorisation)
 * for the slots whose `slot_mask[i] != 0` (all slots if slot_mask == NULL; HOST pointer of
 * max_batch bytes).  Host-synchronous: waits for all work in flight on the device first. */
int cmpc_reset_warm(cmpc_handle* h, const uint8_t* slot_mask);
/* Stream-ordered form for slots [slot0, slot0+B): `slot_mask` is a DEVICE pointer of B bytes (or
 * NULL = all of them); enqueued on `stream`, usable inside a CUDA graph capture. */
int cmpc_reset_warm_async(cmpc_handle* h, int32_t B, int32_t slot0, const uint8_t* slot_mask,
                          void* stream);
/* Copy warm-start forces x [B,N,12] and duals y [B,N,4,3] of slots [slot0, slot0+B)
 * to / from DEVICE buffers (y may be NULL). */
int cmpc_get_warm(cmpc_handle* h, int32_t B, int32_t slot0, float* x, float* y, void* stream);
int cmpc_set_warm(cmpc_handle* h, int32_t B, int32_t slot0, const float* x, const float* y,
                  void* stream);

/* Rigid-body parameters of slots [slot0, slot0+B): mass [B] (kg) and the body-frame inverse inertia
 * ibody_inv [B,3,3] (row-major, symmetric), DEVICE pointers.  Stream-ordered on `stream`, usable inside a
 * graph capture; the data is read on the device only, never on the host.
 *  - A body belongs to a problem slot, like the warm-start state, and stays until it is set again (bodies
 *    change at episode resets, not every tick).  Every entry point that solves or evaluates slot s uses
 *    slot s's body: cmpc_solve, cmpc_solve_host (zero-copy and staged), cmpc_solve_host_async and the
 *    hardest-first launch order.  cmpc_condense and cmpc_plant_step take no slot0: problem / robot i uses
 *    slot i, i.e. slots [0, B).
 *  - A slot never given a body uses the configuration's (cfg.mass, diag(cfg.ibody_inv)); this holds on
 *    every stream, the handle fills all slots at cmpc_create.
 *  - After the first successful call the handle launches the body-reading instantiations of its solve
 *    kernels for all of its slots (a handle that never calls it launches the kernels it always did).
 *    There is no way back; setting the configuration's values again gives the same answers.  A CUDA
 *    graph captured before the first call keeps the kernels it captured.
 *  - The factorisation-cache entries of the written slots are invalidated by the same stream-ordered
 *    work that writes the bodies (the cached factor depends on the body).
 *  - A slot whose mass is not finite and positive, or whose ibody_inv has a non-finite entry, is stored
 *    so that every later solve of it reports CMPC_STATUS_NAN; other slots are unaffected.
 *  - Layout on the device: per slot 12 floats {1/m, ibody_inv row-major (9), 0, 0}, read by a CTA as
 *    three 16-byte loads.
 * CMPC_ERR_INVALID for a null handle or pointer or a slot range outside max_batch (the device is not
 * touched).  Available from the 0.3 series on; detect it by its symbol. */
int cmpc_set_body(cmpc_handle* h, int32_t B, int32_t slot0, const float* mass, const float* ibody_inv,
                  void* stream);

/* Contact surfaces of slots [slot0, slot0+B), per leg and stage of the handle's horizon N, DEVICE pointers (all
 * four required): normal [B,N,4,3], the outward ground normal under leg l at stage i (any length), and mu, f_min,
 * f_max [B,N,4].
 *  - Contact frame: n = normal/|normal|; t1 = normalise(e_x - n_x n) if n_x^2 <= 1/2, else
 *    normalise(e_y - n_y n); t2 = n x t1.  For normal = (0,0,c), c > 0, this is exactly the world axes.  The
 *    leg-stage's force f is kept in {f : f.n in [f_min, f_max], |f.t1| <= mu f.n, |f.t2| <= mu f.n}, the
 *    world-axis friction frustum rotated onto the surface.
 *  - A contact belongs to a problem slot, like the warm-start state and the body, and stays until it is set
 *    again.  Every entry point that solves slot s uses it: cmpc_solve, cmpc_solve_host (zero-copy and staged)
 *    and cmpc_solve_host_async.  For such a slot the solve's mu[b] is not used by the solve (the hardest-first
 *    launch order still scores with it, which changes the order, never the answers).
 *  - A slot never given a contact keeps the world axes, the call's mu[b] and cfg.f_min / cfg.f_max, on every
 *    stream.
 *  - Storage (32 B per leg-stage: {n, mu}, {f_min, f_max, 0, 0}, at the kernel horizon's stride on a padded
 *    horizon, whose padding stages are all-swing) is allocated by the first call.  That call initialises every
 *    slot host-synchronously on `stream` before it enqueues the copy, so it cannot be captured: inside a stream
 *    capture it returns CMPC_ERR_INVALID before any CUDA work, and the capture stays valid.  Later calls are
 *    stream-ordered and usable inside a graph capture.
 *  - After the first successful call the handle launches the contact-reading instantiations of its solve kernels
 *    for all of its slots (with the configuration's body where no cmpc_set_body was made); setting flat contacts
 *    with the call's mu and the configuration's bounds gives the same answers as no contact.  A CUDA graph
 *    captured before the first call keeps the kernels it captured.
 *  - Factorisation-cache entries stay valid: the cached factor does not depend on the constraint set.
 *  - A leg-stage whose normal is non-finite or shorter than 1e-6, whose mu is non-finite or negative, or whose
 *    bounds are non-finite or violate 0 <= f_min <= f_max is stored so that every later solve of its slot
 *    reports CMPC_STATUS_NAN; other slots are unaffected.
 *  - cmpc_condense and cmpc_plant_step do not use contacts.
 * CMPC_ERR_INVALID for a null handle or pointer, B < 0 or a slot range outside max_batch (the device is not
 * touched).  Available from the 0.3 series on; detect it by its symbol. */
int cmpc_set_contact(cmpc_handle* h, int32_t B, int32_t slot0, const float* normal, const float* mu,
                     const float* f_min, const float* f_max, void* stream);

/* Cost weights of slots [slot0, slot0+B), DEVICE pointers (both required): w [B,13], the state weights in the
 * layout of cfg.w, and r_weight [B], the force weight of cfg.r_weight.
 *  - Weights belong to a problem slot, like the warm-start state, the body and the contact, and stay until they
 *    are set again.  Every entry point that solves slot s uses them: cmpc_solve, cmpc_solve_host (zero-copy and
 *    staged) and cmpc_solve_host_async; the hardest-first launch order scores with them (which changes the order,
 *    never the answers).  cmpc_condense takes no slot0: problem i uses slot i, i.e. slots [0, B).
 *    cmpc_plant_step, cmpc_assemble and the leg functions do not use weights.
 *  - A slot never given weights keeps cfg.w / cfg.r_weight, on every stream.
 *  - Storage is allocated by the first call: per slot 64 B {w[0..12], r_weight, 0, 0} and, for kernel horizons
 *    NK <= 30 (those with a dense or condense kernel), the slot's horizon Gram matrices M^-1 and M, 6 NK^2 floats
 *    each (blockdiag(M_N, I) on a padded horizon).  That is 4.8 KB per slot at N = 10 (20 MB for 4096 slots) and
 *    43 KB at N = 30 (0.7 GB for 16384 slots); N > 30 keeps the 64 B only.  The first call initialises every
 *    slot host-synchronously on `stream` from the handle's own Gram matrices and configuration before it enqueues
 *    the store, so it cannot be captured: inside a stream capture it returns CMPC_ERR_INVALID before any CUDA
 *    work, and the capture stays valid.  Later calls are stream-ordered and usable inside a graph capture.
 *  - The store builds each slot's Gram matrices on the device in fp64 in the operation order of cmpc_create and
 *    rounds them to fp32: the configuration's weights give exactly the handle's matrices, and the same answers as
 *    a slot never given weights.
 *  - After the first successful call the handle launches the weight-reading instantiations of its solve kernels
 *    for all of its slots (with the configuration's body where no cmpc_set_body was made).  A CUDA graph captured
 *    before the first call keeps the kernels it captured.
 *  - The factorisation-cache entries of the written slots are invalidated by the same stream-ordered work that
 *    writes the weights (the cached factor depends on M^-1 and r_weight).
 *  - A slot is stored so that every later solve of it reports CMPC_STATUS_NAN, other slots being unaffected, when
 *    an entry of w is non-finite or negative, w[6] != w[7] (what cmpc_create reports as CMPC_ERR_UNSUPPORTED), the
 *    Gram matrix of an axis fails cmpc_create's positive-pivot test (a zero velocity-like weight w[6 + a] always
 *    does, e.g. both weights of an axis zero), or r_weight is non-finite or negative.
 * CMPC_ERR_INVALID for a null handle or pointer, B < 0 or a slot range outside max_batch (the device is not
 * touched).  Available from the 0.3 series on; detect it by its symbol. */
int cmpc_set_weights(cmpc_handle* h, int32_t B, int32_t slot0, const float* w, const float* r_weight, void* stream);

/* Known external wrench on the trunk of slots [slot0, slot0+B), per stage of the handle's horizon N, DEVICE pointers
 * (both required): force [B,N,3], the external force on the trunk, and torque [B,N,3], the external torque about the
 * CoM, both in the world frame (a force F applied at a point p is the torque (p - com) x F).  A towed load, a tether,
 * wind or a disturbance observer's estimate enters the model as the affine term it is instead of an unmodelled
 * disturbance.
 *  - A wrench belongs to a problem slot, like the warm-start state, the body, the contact and the weights, and stays
 *    until it is set again.  Every entry point that solves slot s uses it: cmpc_solve, cmpc_solve_host (zero-copy and
 *    staged) and cmpc_solve_host_async.  cmpc_condense and cmpc_plant_step take no slot0: problem / robot i uses
 *    slot i, i.e. slots [0, B); the plant applies stage 0 of robot i's wrench.  cmpc_assemble, the leg functions and
 *    the hardest-first launch order do not use it.
 *  - A slot never given a wrench has zero wrench, on every stream.
 *  - The wrench changes only the free response of x0, by its forced response phi (the wrench integrated like the
 *    leg forces, with the slot's body and yaw x0[2] frozen over the horizon): the QP with the wrench is the QP without
 *    it on x_des - phi, and its predicted states are that QP's X + phi.  A solve of a handle with wrenches runs the
 *    same solve kernels as one without, plus a kernel before the solve that writes x_des - phi to a per-slot copy and,
 *    when X or status is requested, one after it that adds phi to X: cmpc_launch_count grows by at most 2 per solve.
 *    A zero wrench gives the same answers, bit for bit, as no wrench.
 *  - Storage is allocated by the first call: per slot 24 N bytes for the wrenches (240 B at N = 10) and, when N has
 *    its own compiled kernel, 52 (N + 1) bytes for the shifted x_des (a padded horizon shifts its padded copy).  That
 *    call zero-fills every slot host-synchronously on `stream` before it enqueues the store, so it cannot be captured:
 *    inside a stream capture it returns CMPC_ERR_INVALID before any CUDA work, and the capture stays valid.  Later
 *    calls are stream-ordered and usable inside a graph capture.
 *  - Factorisation-cache entries stay valid: the cached factor does not depend on x_des.
 *  - A slot with a non-finite entry is stored so that every later solve of it reports CMPC_STATUS_NAN, an all-swing
 *    problem included; other slots are unaffected.
 * CMPC_ERR_INVALID for a null handle or pointer, B < 0 or a slot range outside max_batch (the device is not
 * touched).  Available from the 0.3 series on; detect it by its symbol. */
int cmpc_set_wrench(cmpc_handle* h, int32_t B, int32_t slot0, const float* force, const float* torque, void* stream);

/* Force references of slots [slot0, slot0+B), per leg and stage of the handle's horizon N, DEVICE pointers (both
 * required): f_ref [B,N,4,3], the ground-reaction force wanted from leg l at stage i (world frame, the force on the
 * robot, like U), and weight [B,N,4], its weight w_f >= 0.  The objective gains sum over stance leg-stages of
 * w_f ||f - f_ref||^2 (in condensed form H += 2 w_f, g -= 2 w_f f_ref on the stance forces), on top of the slot's
 * r_weight ||u||^2.  A policy's desired forces, a planner's force plan, a load-sharing prior or a soft derating of
 * one leg (f_ref = 0 with a large weight; f_max of cmpc_set_contact is the hard form) enter the QP this way.
 *  - References belong to a problem slot, like the warm-start state, the body, the contact, the weights and the
 *    wrench, and stay until they are set again.  Every entry point that solves slot s uses them: cmpc_solve,
 *    cmpc_solve_host (zero-copy and staged) and cmpc_solve_host_async.  cmpc_condense takes no slot0: problem i uses
 *    slot i, i.e. slots [0, B).  The hardest-first launch order, cmpc_plant_step, cmpc_assemble and the leg
 *    functions do not use them (for the launch order this changes the order, never the answers).
 *  - A slot never given references has zero weight, on every stream.  Swing leg-stages ignore their entries.
 *  - A zero weight gives the same answers, bit for bit, as a handle that never called this, whatever f_ref holds.
 *  - Storage is allocated by the first call: 16 B per leg-stage {f_ref, w_f} at the kernel horizon's stride (640 B
 *    per slot at N = 10; the padding stages of a padded horizon are zero).  The kernels that read references are
 *    compiled with per-slot weights: on a handle that never called cmpc_set_weights the first call also allocates
 *    and fills the weight storage as the first cmpc_set_weights does, with the configuration's weights in every
 *    slot (which give the same answers as the configuration's weights; 4.8 KB per slot at N = 10 and 43 KB at
 *    N = 30, 0.7 GB for 16384 slots).  The first call initialises every slot host-synchronously on `stream` before
 *    it enqueues the store, so it cannot be captured: inside a stream capture it returns CMPC_ERR_INVALID before any
 *    CUDA work, and the capture stays valid.  Later calls are stream-ordered and usable inside a graph capture.
 *  - After the first successful call the handle launches the reference-reading instantiations of its solve kernels
 *    for all of its slots (with the configuration's body where no cmpc_set_body was made).  cmpc_launch_count per
 *    solve does not change.  A CUDA graph captured before the first call keeps the kernels it captured.
 *  - The factorisation-cache entries of the written slots are invalidated by the same stream-ordered work that
 *    writes the references (the cached factor depends on each leg's 1/(sigma + rho + 2 r_weight + 2 w_f)).
 *  - A slot with a non-finite f_ref entry, or a non-finite or negative weight, on any leg-stage (swing ones
 *    included) is stored so that every later solve of it reports CMPC_STATUS_NAN, an all-swing problem included;
 *    other slots are unaffected.
 * CMPC_ERR_INVALID for a null handle or pointer, B < 0 or a slot range outside max_batch (the device is not
 * touched).  Available from the 0.3 series on; detect it by its symbol. */
int cmpc_set_force_ref(cmpc_handle* h, int32_t B, int32_t slot0, const float* f_ref, const float* weight,
                       void* stream);

/* Stage weights of slots [slot0, slot0+B), DEVICE pointers (both required): w [B,N,13], the state weights of every
 * stage of the handle's horizon N, and r_weight [B], the force weight of cfg.r_weight.  Row i of w[b] weighs the
 * predicted state X[b, i+1] in the layout of cfg.w; row N-1 is the terminal weight.  A heavier terminal weight
 * standing in for the cost beyond a short horizon, ramped or discounted tracking, weights that follow the gait or
 * randomised per-stage gains enter the QP this way.
 *  - Stage weights belong to a problem slot, like the warm-start state, the body, the contact, the weights, the
 *    wrench and the force references, and stay until they are set again.  Every entry point that solves slot s uses
 *    them: cmpc_solve, cmpc_solve_host (zero-copy and staged) and cmpc_solve_host_async; the hardest-first launch
 *    order scores with them (which changes the order, never the answers).  cmpc_condense takes no slot0: problem i
 *    uses slot i, i.e. slots [0, B).  cmpc_plant_step, cmpc_assemble and the leg functions do not use them.
 *  - One source of truth: once a handle has stage weights, its kernels read the stage weights of every slot, and a
 *    later cmpc_set_weights(w, r_weight) writes its w into every stage of the slots it covers.
 *    cmpc_set_weights(w, r) and cmpc_set_stage_weights(w repeated N times, r) give the same state.
 *  - The same w on every stage gives the same answers, bit for bit, as cmpc_set_weights(w, r_weight) on the same
 *    handle configuration, and the configuration's weights on every stage those of a handle that never set weights.
 *  - Storage is allocated by the first call: 48 B per stage (w[0..11]) at the kernel horizon's stride (480 B per slot
 *    at N = 10, 2.9 KB at N = 60; the padding stages of a padded horizon are zero and carry no cost).  The first call
 *    gives every stage of every slot that slot's current weights (the configuration's, or those of an earlier
 *    cmpc_set_weights).  The kernels that read stage weights are compiled with per-slot weights and force references:
 *    on a handle that never called cmpc_set_weights the first call also allocates and fills the weight storage as
 *    the first cmpc_set_weights does, and on one that never called cmpc_set_force_ref the reference storage with zero
 *    weight (both give the answers of no such call).  The first call initialises every slot host-synchronously on
 *    `stream` before it enqueues the store, so it cannot be captured: inside a stream capture it returns
 *    CMPC_ERR_INVALID before any CUDA work, and the capture stays valid.  Later calls are stream-ordered and usable
 *    inside a graph capture.
 *  - The store builds each slot's Gram matrices from the stage weights on the device, in fp64 in the operation order
 *    of cmpc_create, M_a[j][j'] = 2 sum_{k > max(j,j')} (w_pos,a,k dt^4 (k-1-j)(k-1-j') + w_vel,a,k dt^2).
 *  - After the first successful call the handle launches the stage-weight-reading instantiations of its solve
 *    kernels for all of its slots (with the configuration's body where no cmpc_set_body was made).
 *    cmpc_launch_count per solve does not change.  A CUDA graph captured before the first call keeps the kernels it
 *    captured.
 *  - The factorisation-cache entries of the written slots are invalidated by the same stream-ordered work that
 *    writes the weights (the cached factor depends on M^-1).
 *  - A slot is stored so that every later solve of it reports CMPC_STATUS_NAN, other slots being unaffected, when
 *    an entry of w on some stage is non-finite or negative, w[i][6] != w[i][7] on some stage i, the Gram matrix of an
 *    axis fails cmpc_create's positive-pivot test (a zero terminal velocity-like weight w[N-1][6 + a] always does:
 *    the last row of M_a is then 2 w_vel,N dt^2), or r_weight is non-finite or negative.
 * CMPC_ERR_INVALID for a null handle or pointer, B < 0 or a slot range outside max_batch (the device is not
 * touched).  Available from the 0.3 series on; detect it by its symbol. */
int cmpc_set_stage_weights(cmpc_handle* h, int32_t B, int32_t slot0, const float* w, const float* r_weight,
                           void* stream);

/* ---- on-device parameter assembly and closed-loop plant (SURVEY.md section 8f) ------------
 * Per-robot gait tables, all DEVICE pointers: the arrays of reference FootstepPlanner.plan
 * (src/footstep_planner.py:72-177) plus the reference velocities of src/main.py:31-46. */
typedef struct cmpc_gait_tables {
  const float* plan_pos;    /* [B,S,4,3] planned footholds per step                        */
  const uint8_t* feet_id;   /* [B,S] stance bits of each step's single-support part        */
  const int32_t* ss;        /* [B] single-support ticks                                    */
  const int32_t* ds;        /* [B] double-support ticks                                    */
  const float* v_ref;       /* [B,3]                                                       */
  const float* omega_ref;   /* [B]                                                         */
  const float* rp0;         /* [B,2] initial roll, pitch (src/mpc.py:203)                  */
  int32_t S;                /* steps in the plan                                           */
  int32_t total_steps;      /* params['total_steps'] (src/mpc.py:181)                      */
  float step_height;        /* src/foot_trajectory_generator.py:23                         */
  float g;                  /* params['g']                                                 */
} cmpc_gait_tables;

/* Replaces the Python parameter loops of MPC.solve (src/mpc.py:178-255) for B robots at the
 * tick stored in `tick` (device int32): writes x_des [B,N+1,13], r [B,N,4,3], mask [B,N].
 * x [B,13] measured state, yaw_start [B] / com_start [B,3] reference accumulators. */
int cmpc_assemble(cmpc_handle* h, int32_t B, const cmpc_gait_tables* gt, const int32_t* tick,
                  const float* x, const float* yaw_start, const float* com_start, float* x_des,
                  float* r, uint8_t* mask, void* stream);

/* Closed-loop plant for BASELINE config 5 (DART is unavailable: single-rigid-body forward
 * Euler with the applied first-stage forces U[:,0,:] and the true lever arms r[:,0]; robot i
 * has the body of slot i, see cmpc_set_body, and stage 0 of the external wrench of slot i, see
 * cmpc_set_wrench), plus
 * the reference-accumulator advance of src/mpc.py:261-262 and `*tick += 1`.
 * track_err [B,2] accumulates |p-p_des|^2 and |Theta-Theta_des|^2. */
int cmpc_plant_step(cmpc_handle* h, int32_t B, const cmpc_gait_tables* gt, int32_t* tick,
                    float* x, const float* r, const float* U, const float* x_des,
                    float* yaw_start, float* com_start, float* track_err, void* stream);

/* Leg controllers that consume the solve (src/main.py:193-282, SURVEY.md section 8f.3) for B
 * robots at the tick stored in `tick`: stance legs get tau = J'(-f) with f = U[:,0,leg]
 * (ground_controller, src/main.py:203-214), swing legs the PD + feed-forward law of
 * swing_leg_controller (src/main.py:219-282) on the swing reference of
 * src/foot_trajectory_generator.py:27-96.  Which legs are stance follows src/main.py:152-160.
 * DEVICE pointers: U [B,N,12]; J, Jdot, Mleg [B,4,3,3] (the leg's 3x3 blocks of DART's
 * getLinearJacobian / getJacobianClassicDeriv[3:] / getMassMatrix()[3:6]); cg, dq, foot_pos,
 * foot_vel [B,4,3]; outputs tau [B,4,3], p_des [B,4,3] (nullable, the desired foot position
 * the reference logs), stance [B] uint8 bits (nullable).  kp, kd: HOST pointers to the 3
 * diagonal gains (reference: 250, 15). */
int cmpc_leg_torques(cmpc_handle* h, int32_t B, const cmpc_gait_tables* gt, const int32_t* tick,
                     const float* U, const float* J, const float* Jdot, const float* Mleg,
                     const float* cg, const float* dq, const float* foot_pos, const float* foot_vel,
                     const float* kp, const float* kd, float* tau, float* p_des, uint8_t* stance,
                     void* stream);

/* Lite3 leg kinematics for B robots (SURVEY.md section 8f.3): everything cmpc_leg_torques needs that
 * the reference reads from DART (src/main.py:203-214, 236-262, 286-350), in closed form from the
 * joint tree of lite3_urdf/urdf/Lite3.urdf (hip offsets :45, thigh offset :73, link lengths :100,
 * :122, axes :48, :76, :103, link masses / centres of mass).  DEVICE pointers: base_pos, theta
 * (torso rotation vector = retrieve_state()['TORSO']['pos']), v_base, w_base [B,3] (world frame);
 * q, dq [B,4,3] (HipX, HipY, Knee of FL, FR, HL, HR).  Outputs: foot_pos, foot_vel [B,4,3]; J, Jdot
 * [B,4,3,3] world-frame linear Jacobian of the foot w.r.t. the leg's joints and its time derivative
 * (getLinearJacobian / getJacobianClassicDeriv[3:] at the leg's columns); Mleg [B,4,3,3] =
 * sum_i m_i J_com_i, the base-translation rows of the joint-space inertia matrix at the leg's
 * columns (getMassMatrix()[3:6]); cg [B,4,3] gravity torques of the leg's joints (the velocity-product
 * part of getCoriolisAndGravityForces is not modelled).  Mleg, cg may be NULL. */
int cmpc_leg_kinematics(cmpc_handle* h, int32_t B, const float* base_pos, const float* theta,
                        const float* v_base, const float* w_base, const float* q, const float* dq,
                        float* foot_pos, float* foot_vel, float* J, float* Jdot, float* Mleg, float* cg,
                        float gravity, void* stream);

/* Measures the FP32 FMA throughput of `device` (TFLOP/s, best of 4 timed launches of an 8-chain
 * FMA kernel): the denominator of the on-chip roofline of the solve kernel. */
int cmpc_fp32_peak(int32_t device, float* tflops);

/* Running totals of a rollout, one launch: acc[0] += sum(iters), acc[1] += #(status != solved),
 * acc[2] += factorisation-cache hits of slots [slot0, slot0+B) in the last solve (0 without the
 * cache).  iters, status [B] and acc [3] (64-bit unsigned) are DEVICE pointers. */
int cmpc_accumulate_stats(cmpc_handle* h, int32_t B, int32_t slot0, const int32_t* iters,
                          const int32_t* status, uint64_t* acc, void* stream);

/* Factorisation-cache bookkeeping of slots [slot0, slot0+B) (cfg.cache_factorization): copies
 * meta [B,4] = {rho of the cached factor, yaw it was computed at, valid (0/1), reused by the
 * last cmpc_solve (0/1)} to a DEVICE buffer. */
int cmpc_get_cache_meta(cmpc_handle* h, int32_t B, int32_t slot0, float* meta, void* stream);

/* Duration in ms of the solve kernel of the most recent cmpc_solve (cfg.time_kernel = 1):
 * CUDA events recorded on the launching stream immediately around that one kernel, i.e. without
 * the two scheduling kernels in front of it.  Synchronises on the closing event. */
int cmpc_last_kernel_ms(cmpc_handle* h, float* ms);

/* Number of kernels this library has launched on behalf of `h` since creation (a solve of a
 * handle with wrenches launches up to 2 more, see cmpc_set_wrench). */
int64_t cmpc_launch_count(const cmpc_handle* h);

/* Horizons with their own compiled kernel: writes up to `cap` values, returns the count. */
int cmpc_supported_horizons(int32_t* out, int32_t cap);
/* Largest horizon a handle can be created for; the compiled horizon that horizon N runs on
 * (N itself, or the next larger compiled one; negative error code outside 1..max). */
int cmpc_max_horizon(void);
int cmpc_kernel_horizon(int32_t N);
/* 1 if kernel `variant` (cfg.kernel_variant: 0 or 5) is compiled for the kernel horizon of N. */
int cmpc_has_variant(int32_t N, int32_t variant);

int cmpc_version(void);               /* major*1000 + minor */
const char* cmpc_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* CMPC_H */
