/* mpcb200.h -- C ABI of the B200-native MPC inner loop (libmpcb200.so).
 *
 * Drop-in boundary for ONE path of ShittyWizard/DiplomJourney: expansion of the
 * control-input tree over the horizon, kinematic-bicycle rollout of every
 * candidate control sequence, terminal tracking cost, first-minimum argmin.
 * The reference has no FFI of its own; the functions below replace the bodies
 * of the Python functions cited on each entry (paths are into the reference
 * repository).  Plain C: pointers + sizes, no torch types, no exceptions.
 *
 * Conventions
 *   - every function returns 0 (MPCB_OK) or a negative mpcb_status; the text
 *     of the last error of a handle is available from mpcb_last_error().
 *   - control c = iv*nb + ib (velocity outer loop, angle inner loop:
 *     math_model.py:163-164).  S = nv*nb controls per step.
 *   - FULL leaf index  j = sum_k i_k * S^(H-1-k), i_0 = first applied control
 *     (math_model.py:159-200).  HELD leaf index k in [0,S): control k held for
 *     all H steps (math_model_tree.py:308-361, CoordinateTree.py:20-30).
 *   - ties resolve to the lowest leaf index (strict '<', math_model.py:195).
 *   - a handle owns one device, one stream and its scratch; it is not
 *     thread-safe, distinct handles are independent.
 *   - "_host" entry points take host pointers and copy; "_device" entry points
 *     take device pointers valid on the handle's device and enqueue on the
 *     handle's stream without synchronising (call mpcb_sync).
 *   - there is no CPU fallback: without a CUDA device mpcb_create fails.
 */
#ifndef MPCB200_H
#define MPCB200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define MPCB_API __attribute__((visibility("default")))
#else
#define MPCB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mpcb_handle_s mpcb_handle;

typedef enum {
    MPCB_OK = 0,
    MPCB_ERR_INVALID = -1,      /* bad argument (null pointer, H out of range, ...) */
    MPCB_ERR_CUDA = -2,         /* CUDA runtime error, see mpcb_last_error */
    MPCB_ERR_NO_GRID = -3,      /* solve before mpcb_set_grid */
    MPCB_ERR_EMPTY_GRID = -4,   /* mpcb_set_grid with nv == 0 or nb == 0: a tree without candidates (the reference's loops then
                                   simply do not execute and the previous trajectory is returned, math_model_tree.py:308-361) */
    MPCB_ERR_TOO_LARGE = -5,    /* S^H does not fit in int64 */
    MPCB_ERR_NO_DEVICE = -6,
    MPCB_ERR_NCCL = -7
} mpcb_status;

/* tree semantics */
#define MPCB_MODE_FULL 0 /* predictive_control, math_model.py:136-231 / run_math_model.py:133-228 */
#define MPCB_MODE_HELD 1 /* predictive_control, math_model_tree.py:278-496 (CoordinateTree-pruned) */
/* terminal cost */
#define MPCB_COST_MM 0   /* control_criterion math_model.py:82-86:  1e4 d + 10 (atan(x_t/y_t)-phi)^2 + 100 d_l^2 */
#define MPCB_COST_TREE 1 /* control_criterion math_model_tree.py:82-87: 1e4 d + 1e4 d_l^2 */
/* expansion algorithm (FULL only; HELD always walks one thread per leaf) */
#define MPCB_ALGO_AUTO 0
#define MPCB_ALGO_LEAFWALK 1 /* one thread per leaf walks the whole horizon (2H+1 MUFU per rollout) */
#define MPCB_ALGO_PREFIX 2   /* one thread per depth-(H-1) node, loops its S children (prefix sharing) */

#define MPCB_MAX_H 8

/* per-solve flags (uint8 per solve) */
#define MPCB_FLAG_SLOW 1 /* steps_for_slowing > 0: every velocity := max(min(V), v_min), math_model_tree.py:312-316;
                            honoured by HELD solves only (the FULL scripts have no slow-down) */
#define MPCB_FLAG_SKIP 2 /* do not solve this entry (a robot of a batch that has already stopped): index -1, cost NaN */

MPCB_API int mpcb_version(void);
MPCB_API int mpcb_device_count(void);

MPCB_API int mpcb_create(int device_ordinal, mpcb_handle **out);
MPCB_API int mpcb_destroy(mpcb_handle *h);
MPCB_API const char *mpcb_last_error(const mpcb_handle *h);
/* the CUDA stream (cudaStream_t) the handle enqueues on, as an opaque pointer */
MPCB_API void *mpcb_stream(mpcb_handle *h);
MPCB_API int mpcb_sync(mpcb_handle *h);

/* Control grid + vehicle constants.  Replaces the module-level grids
 * (math_model.py:23-30) / the per-tick windows handed to predictive_control
 * (math_model_tree.py:543-551) and builds the per-control tables
 * dphi_c = (v_c/L) tan(beta_c) delta_t, s_c = v_c delta_t   (math_model.py:69-78,90-114). */
MPCB_API int mpcb_set_grid(mpcb_handle *h, const double *v, int nv, const double *beta, int nb,
                  double L, double delta_t, double v_min);

/* Options: "tol_scale" (candidate-window multiplier, default 1), "algo" (MPCB_ALGO_*),
 * "refine" (1 = float64 re-evaluation of near-minimal leaves, default; 0 = fp32 winner),
 * "small_path" (1 = host-API HELD solves with <= 4096 candidates run as one float64 launch, default),
 * "zero_copy" (1, default: on that path, up to 64 solves read their inputs from and write their results to mapped
 * pinned host memory -- one launch and one synchronisation per call, no copy; 0 = one staged copy each way),
 * "prune" (1 = exact branch-and-bound in the prefix kernel: depth-(H-1) nodes whose children provably cannot
 * reach the refinement window of the best leaf are skipped -- a lower bound from the distance to the target, the
 * steering and speed limits and the most favourable line / heading offsets against the best cost found so far;
 * identical results; default 1, 0 = evaluate every leaf as the reference does),
 * "subtree_cut" (with prune and H >= 3; identical results in every mode.  1: every 256-node tile is tested against
 * the bound of its depth-(H-2) node(s) before any of its nodes is set up; fully asynchronous.  3: the frontier of
 * subtrees that may still hold the argmin is expanded level by level from the root with a bound over all leaves below
 * each node, and only the children of the depth-(H-2) survivors are ever set up; the call then synchronises the stream
 * once to read whether a frontier outgrew "frontier_cap" entries (default 2^22), in which case mode 1 redoes pass 1.
 * 2, default: mode 3 for trees of more than 2^23 tiles per call, mode 1 otherwise.  0: node-level cut only),
 * "screen" (exhaustive prefix pass 1, i.e. prune = 0; identical results.  1: every leaf's cost terms -- scaled
 * squared distance dd, line offset q, heading offset gg -- are formed, but the MUFU.SQRT that turns them into the value
 * sqrt(dd) + q^2 + gg^2 is only spent in nodes holding a leaf that can still matter: with cn the largest value a leaf
 * of the node may have and still beat the solve's upper bound (an exact probe of the S held sequences, tightened by
 * every node that found something), a leaf matters iff t = cn - q^2 - gg^2 > 0 and fma(t, t, -dd) > 0; such nodes are
 * re-run with the square roots.  2, default: the same screen in two stages -- every leaf's dd first, with a per-node
 * bound on q^2 + gg^2 in place of the leaf's own terms; only the nodes that pass go through the screen of 1, and the
 * nodes the screen flags are exactly those of 1 (grids whose row table does not fit one shared-memory chunk run 1).
 * 0: one MUFU.SQRT per leaf, no upper bound involved),
 * "prefilter" (1, default; identical results: in the pruned pass 1 a node's bound is first evaluated in fp32 from an fp32
 * walk and the node dropped if that exceeds the upper bound by a margin of 8 error bounds -- which the float64 test would
 * do as well -- so that the float64 set-up is only paid by nodes near the bound; 0 = float64 test for every node),
 * "candidate_list" (entries; identical results: the refinement pass lists the leaves whose fp32 value lies inside the
 * error window and a second kernel evaluates them in float64 one thread each; candidates beyond the capacity -- or all of
 * them with 0 -- are evaluated by the thread that found them.  Default -1 = automatic: 2^20 for the leafwalk algorithm,
 * none for the prefix algorithm while it has a "node_list", whose scan evaluates an in-window leaf from its node's
 * float64 pose with one step),
 * "node_list" (entries, default 2^15; identical results: the refinement pass first lists the depth-(H-1) nodes whose
 * bound reaches into the error window and a second kernel scans the leaves of each listed node with one warp, so that
 * a few thousand scans are spread evenly over the GPU instead of staying with the few warps that found the nodes;
 * nodes beyond the capacity -- or all of them with 0 -- are scanned where they are found, which is as good when there
 * are many),
 * "nodes_per_thread" (1, 2 or 4, default 4: depth-(H-1) nodes each thread of the exhaustive prefix pass 1 holds --
 * identical results; with the two-stage screen four nodes share each table load of its stage-1 loop), "dump_direct" (diagnostics: mpcb_dump_leaves_host returns the cheaper fp32 form pass 1 ranks
 * with instead of the one pass 2 filters with; default 0), "frontier_cap" (see "subtree_cut"). */
MPCB_API int mpcb_set_option(mpcb_handle *h, const char *name, double value);

/* Batch of N independent MPC solves sharing the grid.  Replaces N calls of
 * predictive_control (math_model.py:136 / math_model_tree.py:278).
 *   state[N][3]   x, y, phi at the start of the solve
 *   target[N][2]  x_t, y_t            (module globals in the reference)
 *   origin[N][2]  x_0, y_0 of the tracked line (moves on new_target, math_model_tree.py:119-125)
 *   threshold[N]  accept only a leaf with cost < threshold (optimal_criterion, math_model.py:195);
 *                 NULL = +inf
 *   flags[N]      MPCB_FLAG_*; NULL = 0
 * outputs (any may be NULL):
 *   best_cost[N]        float64 cost of the minimal leaf (reference formula, float64)
 *   best_index[N]       its leaf index, or -1 if no leaf has cost < threshold (or all costs are NaN)
 *   best_traj[N][H][3]  float64 poses after each step of the minimal leaf's sequence
 *   first_control[N][2] (v, beta) of its first step (v after the slow-down override)
 * Restricting FULL to first controls [i0_begin, i0_end) gives one rank's share of a
 * split tree (indices stay global); pass 0, -1 for the whole tree. */
MPCB_API int mpcb_solve_batch_host(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N,
                          const double *state, const double *target, const double *origin,
                          const double *threshold, const uint8_t *flags,
                          int64_t i0_begin, int64_t i0_end,
                          double *best_cost, int64_t *best_index, double *best_traj, double *first_control);

MPCB_API int mpcb_solve_batch_device(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N,
                            const double *state, const double *target, const double *origin,
                            const double *threshold, const uint8_t *flags,
                            int64_t i0_begin, int64_t i0_end,
                            double *best_cost, int64_t *best_index, double *best_traj, double *first_control);

/* One online tick in ONE call: mpcb_set_grid(v, beta, ...) followed by a single HELD solve -- what
 * math_model_tree.predictive_control does per tick with the window lists handed to it (math_model_tree.py:543-551).
 * Host pointers; threshold = +inf accepts every leaf; flags = MPCB_FLAG_*. */
MPCB_API int mpcb_held_tick_host(mpcb_handle *h, const double *v, int nv, const double *beta, int nb,
                        double L, double delta_t, double v_min, int cost_kind, int H,
                        const double *state, const double *target, const double *origin, double threshold, int flags,
                        double *best_cost, int64_t *best_index, double *best_traj, double *first_control);

/* Every leaf of ONE small tree in enumeration order (debug / plots / parity): the
 * reference scatters all leaf positions (math_model.py:192-193,204).
 *   xy[count][2] float32 terminal position, cost[count] float64 = the kernel's own fp32
 *   evaluation of the leaf cost (offset form, see DESIGN.md) re-based to the absolute cost.
 * Host pointers. algo selects which kernel family evaluates the leaves. */
MPCB_API int mpcb_dump_leaves_host(mpcb_handle *h, int mode, int cost_kind, int H, int algo,
                          const double *state, const double *target, const double *origin, uint8_t flags,
                          int64_t leaf_begin, int64_t count, float *xy, double *cost);

/* Statistics of the last solve on this handle (for tests and bench accounting). */
typedef struct {
    int64_t units;            /* leaves (leafwalk) or depth-(H-1) nodes (prefix) per solve */
    int64_t leaves_per_solve;
    int64_t segments;         /* pass-1 partial minima */
    int64_t refine_segments;  /* segments re-run by the float64 refinement pass */
    int64_t refine_candidates;/* leaves re-evaluated in float64 */
    int64_t pruned_units;     /* depth-(H-1) nodes (x N solves) skipped by the exact branch-and-bound */
    int32_t algo;             /* MPCB_ALGO_* actually used */
    int32_t kernel_launches;  /* kernels enqueued by the last solve */
    int64_t stage2_units;     /* depth-(H-1) nodes (x N solves) that passed stage 1 of the two-stage screen ("screen" 2, row
                                 table), i.e. whose line and heading terms were formed leaf by leaf; 0 otherwise */
} mpcb_stats;
MPCB_API int mpcb_get_stats(mpcb_handle *h, mpcb_stats *out);

/* Device-resident closed loop of the online (HELD) controller for a batch of robots: the tick loop
 * of math_mpc(initial, target, isActual=False) (math_model_tree.py:515-579, without the scripted
 * operator events of the demo run) -- windows vector_of_velocities / vector_of_beta_angles
 * (math_model_tree.py:239-256), HELD solve with the slow-down override (:308-361), finishing
 * heuristic and threshold reset (:388-429), is_on_target and repeated-position stop (:542,559-563) --
 * executed entirely on the GPU, one CTA per robot, float64 throughout.
 * The host computes the window constants exactly as the reference does and passes them in. */
typedef struct {
    double L, delta_t;
    double delta_v, delta_beta;
    double v_max, v_min;
    double beta_limit;      /* beta_max + radians(eps_beta)                   (math_model_tree.py:254) */
    double half_v;          /* (v_acc_max*delta_t)/delta_v                    (math_model_tree.py:241-243) */
    double half_beta;       /* (degrees(beta_acc_max)*delta_t)/degrees(delta_beta) (:251-253) */
    double eps;             /* is_on_target tolerance on the squared distance (:49) */
    int32_t n_v, n_beta;    /* 1 + 2*int(half_v), 1 + 2*int(half_beta) */
    int32_t cost_kind, H;   /* MPCB_COST_*, horizon (3 in the reference) */
    int32_t max_ticks, reserved;
} mpcb_loop_params;

/* per-robot stop reason */
#define MPCB_LOOP_ON_TARGET 0
#define MPCB_LOOP_STALLED 1    /* the reference's "Recursive error." */
#define MPCB_LOOP_MAX_TICKS 2
#define MPCB_LOOP_NO_LEAF 3    /* first tick found no acceptable leaf (the reference raises IndexError) */

/*   init[N][5]            x, y, phi, v, beta     target[N][2], origin[N][2] as for mpcb_solve_batch
 *   first_threshold[N]    optimal_criterion before the first tick (control_criterion of the line
 *                         origin in the reference, math_model_tree.py:676); NULL = +inf
 *   slow_steps[N]         steps_for_slowing at entry; NULL = 0
 *   out_log[N][max_ticks][5]  the 5-list returned by every tick (x, y, phi, v, beta)
 *   out_ticks[N], out_status[N] */
MPCB_API int mpcb_held_closed_loop_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                               const double *init, const double *target, const double *origin,
                               const double *first_threshold, const int32_t *slow_steps,
                               double *out_log, int32_t *out_ticks, int32_t *out_status);
MPCB_API int mpcb_held_closed_loop_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                 const double *init, const double *target, const double *origin,
                                 const double *first_threshold, const int32_t *slow_steps,
                                 double *out_log, int32_t *out_ticks, int32_t *out_status);

/* The same loop WITH the operator events of the reference's run (math_model_tree.py:564-569: turn_right at tick 60,
 * turn_left at 90, new_target at 110 in the demo) applied on the device between ticks: after the tick whose 1-based
 * number equals `tick`, every running robot gets
 *   MPCB_EVENT_NEW_TARGET  new_target(x, y, phi, a, b, v)     math_model_tree.py:118-129: target := (a, b), the tracked line
 *                          restarts at the robot's pose, slow_down(30 deg) -> 10 slowed ticks
 *   MPCB_EVENT_TURN_LEFT / _RIGHT  turn_left / turn_right(x, y, phi, distance = a, v)   :142-215: a synthetic target from
 *                          the robot's pose, the U-turn radius L / sin(beta_max) (`radius_u_turn`) and the quadrant of
 *                          phi, then new_target and slow_down(90 deg) -> 20 slowed ticks
 * One script for the whole batch; its effect differs per robot because it starts from the robot's own pose.
 *   out_final[N][6]  (nullable) x_t, y_t, x_0, y_0, steps_for_slowing, m when the robot stopped */
typedef struct {
    int32_t tick;   /* 1-based number of the tick after which the event fires */
    int32_t kind;   /* MPCB_EVENT_* */
    double a, b;
} mpcb_loop_event;
#define MPCB_EVENT_NEW_TARGET 1
#define MPCB_EVENT_TURN_LEFT 2
#define MPCB_EVENT_TURN_RIGHT 3
MPCB_API int mpcb_held_closed_loop_events_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                      const double *init, const double *target, const double *origin,
                                      const double *first_threshold, const int32_t *slow_steps,
                                      const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                      double *out_log, int32_t *out_ticks, int32_t *out_status, double *out_final);

/* The same loop as the reference's "actual" run math_mpc(..., True) (math_model_tree.py:580-629): after every tick the
 * applied (v, beta) are perturbed by get_actual_velocity / get_actual_beta_angle (:259-275), drawn from the robot's OWN
 * numpy RandomState -- the legacy MT19937 stream, its random() and masked-rejection randint(), bit for bit.  The noisy
 * values are logged (columns 3-4) and build the next tick's acceleration windows.  Velocity is drawn first, then beta,
 * also on the tick that ends in the repeated-position stop; the on-target, max-ticks and no-leaf stops draw nothing.
 * Events as for mpcb_held_closed_loop_events_host (the reference's actual run adds new_target(2, 3) after tick 1).
 *   rng_state[N][625]  in/out: per robot RandomState.get_state()'s key[624] followed by pos (0..624); on return
 *                      the state the generator has after the robot's draws.  NULL, or a pos outside [0, 624], is
 *                      MPCB_ERR_INVALID (checked before anything is copied). */
MPCB_API int mpcb_held_closed_loop_actual_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                      const double *init, const double *target, const double *origin,
                                      const double *first_threshold, const int32_t *slow_steps,
                                      const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                      uint32_t *rng_state,
                                      double *out_log, int32_t *out_ticks, int32_t *out_status, double *out_final);
/* Device flavour of mpcb_held_closed_loop_actual_host: init, target, origin, first_threshold, slow_steps, rng_state
 * (in/out) and every output are device pointers; the event script stays a host array (configuration, like p: it is
 * checked as the host entries check it and copied into handle scratch).  Enqueued without a sync.  Rows of out_log after
 * a robot's last tick are not written: the caller fills out_log beforehand (the host entry fills it with NaN).  pos is
 * not checked (that would need a copy): any pos >= 624 behaves as 624, because the generator twists before its next
 * draw (a robot that draws nothing hands its record back unchanged).  A null rng_state is MPCB_ERR_INVALID. */
MPCB_API int mpcb_held_closed_loop_actual_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                        const double *init, const double *target, const double *origin,
                                        const double *first_threshold, const int32_t *slow_steps,
                                        const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                        uint32_t *rng_state,
                                        double *out_log, int32_t *out_ticks, int32_t *out_status, double *out_final);
/* The actual run's generators seeded on the device as numpy seeds them (the legacy RandomState(seed), not numpy's
 * Generator): rng_state[N][625] receives, per robot, the key[624] + pos (624) RandomState(...).get_state() hands out.
 *   key_len == 0              keys[N] holds one integer seed per robot: RandomState(keys[n]) (mt19937_seed)
 *   1 <= key_len <= 4096      keys[N][key_len] holds one key per robot: RandomState(keys[n, :]) (mt19937_init_by_array;
 *                             RandomState(5) and RandomState([5]) are different streams)
 * Device pointers, enqueued on the handle's stream without a sync.  Another key_len, N < 0 (or N >= 2^31), or a null
 * pointer with N > 0 is MPCB_ERR_INVALID; N == 0 launches nothing. */
MPCB_API int mpcb_rng_seed_device(mpcb_handle *h, int64_t N, const uint32_t *keys, int32_t key_len, uint32_t *rng_state);
/* mpcb_held_closed_loop_actual_host with the generators seeded on the device from keys / key_len (as for
 * mpcb_rng_seed_device, host pointer) in place of rng_state: no generator state crosses the bus on the way in.
 *   rng_state_out[N][625]  (nullable) the generators' states after the run; NULL = they are not copied back */
MPCB_API int mpcb_held_closed_loop_seeded_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                      const double *init, const double *target, const double *origin,
                                      const double *first_threshold, const int32_t *slow_steps,
                                      const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                      const uint32_t *keys, int32_t key_len, uint32_t *rng_state_out,
                                      double *out_log, int32_t *out_ticks, int32_t *out_status, double *out_final);

/* The actual run with numpy's Generator(PCG64) stream (np.random.default_rng) in place of the legacy RandomState: the
 * same loop, events and draw order as mpcb_held_closed_loop_actual_host (velocity: one random(), then integers(0, 5)
 * under 0.4 m/s, else integers(-100, 10); beta: one random(), then integers(-5, 5)), drawn as numpy's Generator draws
 * them -- random() from one 64-bit output, integers() by Lemire's method on 32-bit draws that keep the unused upper half
 * of a 64-bit output for the next 32-bit draw.
 *   pcg_state[N][6]  in/out: per robot Generator.bit_generator.state as six uint64 words: state >> 64, state mod 2^64,
 *                    inc >> 64, inc mod 2^64, has_uint32, uinteger; on return the state after the robot's draws.  NULL,
 *                    has_uint32 outside {0, 1}, uinteger >= 2^32 or an even inc is MPCB_ERR_INVALID (checked before
 *                    anything is copied). */
MPCB_API int mpcb_held_closed_loop_pcg64_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                     const double *init, const double *target, const double *origin,
                                     const double *first_threshold, const int32_t *slow_steps,
                                     const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                     uint64_t *pcg_state,
                                     double *out_log, int32_t *out_ticks, int32_t *out_status, double *out_final);
/* Device flavour of mpcb_held_closed_loop_pcg64_host, as mpcb_held_closed_loop_actual_device is of the MT19937 entry:
 * device pointers (pcg_state in/out), the event script a host array, enqueued without a sync, out_log rows after a
 * robot's last tick not written.  The records are not checked (that would need a copy).  A null pcg_state is
 * MPCB_ERR_INVALID. */
MPCB_API int mpcb_held_closed_loop_pcg64_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                       const double *init, const double *target, const double *origin,
                                       const double *first_threshold, const int32_t *slow_steps,
                                       const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                       uint64_t *pcg_state,
                                       double *out_log, int32_t *out_ticks, int32_t *out_status, double *out_final);
/* The Generator(PCG64) records seeded on the device as numpy seeds them: pcg_state[N][6] receives, per robot, the state
 * of default_rng(SeedSequence(entropy, spawn_key)) (has_uint32 = uinteger = 0).  SeedSequence works on 32-bit words:
 *   entropy      the entropy's little-endian words (an integer expands into as many words as it needs, 0 into one;
 *                a sequence of integers into the concatenation of theirs); 1 <= entropy_len <= 4096
 *   entropy_stride  0: entropy[entropy_len] is shared by all robots; entropy_len: entropy[N][entropy_len], one row each
 *   spawn_key    [N][spawn_len] the words of each robot's spawn key, 0 <= spawn_len <= 4096 (0: no spawn key, and
 *                spawn_key may be NULL).  SeedSequence(root).spawn(N)[i] has root's entropy and the spawn key
 *                root.spawn_key + (root.n_children_spawned + i,).
 * Device pointers, enqueued on the handle's stream without a sync.  Other lengths or strides, N < 0 (or N >= 2^31), or a
 * null pointer that is needed with N > 0 is MPCB_ERR_INVALID; N == 0 launches nothing. */
MPCB_API int mpcb_pcg64_seed_device(mpcb_handle *h, int64_t N, const uint32_t *entropy, int32_t entropy_len,
                                    int32_t entropy_stride, const uint32_t *spawn_key, int32_t spawn_len,
                                    uint64_t *pcg_state);
/* mpcb_held_closed_loop_pcg64_host with the generators seeded on the device from SeedSequence words (as for
 * mpcb_pcg64_seed_device, host pointers) in place of pcg_state.
 *   pcg_state_out[N][6]  (nullable) the generators' states after the run; NULL = they are not copied back */
MPCB_API int mpcb_held_closed_loop_pcg64_seeded_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                            const double *init, const double *target, const double *origin,
                                            const double *first_threshold, const int32_t *slow_steps,
                                            const mpcb_loop_event *events, int32_t n_events, double radius_u_turn,
                                            const uint32_t *entropy, int32_t entropy_len, int32_t entropy_stride,
                                            const uint32_t *spawn_key, int32_t spawn_len, uint64_t *pcg_state_out,
                                            double *out_log, int32_t *out_ticks, int32_t *out_status,
                                            double *out_final);

/* ONE online tick for a batch of robots that each have their OWN acceleration window (SURVEY 8f row f2).  The
 * reference rebuilds the control window per robot and per tick around the robot's current (v, beta)
 * (vector_of_velocities / vector_of_beta_angles, math_model_tree.py:239-256, called at :543-545 and -- with the noisy
 * actuator values of the "actual" run -- at :590-597), so a batch of robots shares no grid and mpcb_set_grid does not
 * apply: the windows are built on the device from `v_beta` with the same float64 expressions, then every robot's
 * HELD tree (math_model_tree.py:308-361) is solved in float64, one CTA per robot, ONE launch for the batch.
 *   p               window constants and horizon (max_ticks is ignored)
 *   state[N][3], v_beta[N][2] = current (v, beta) of each robot, target[N][2], origin[N][2]
 *   threshold[N]    NULL = +inf;  flags[N]  MPCB_FLAG_SLOW / MPCB_FLAG_SKIP, NULL = 0
 * outputs (any may be NULL): as mpcb_solve_batch_*, with best_index = iv * nB + ib inside the robot's own window and
 *   window_shape[N][2] = (nV, nB) of that window.  An empty window (nV == 0 or nB == 0) has no candidate: index -1,
 *   cost NaN -- the reference then finds no improving leaf and hands back the previous trajectory. */
MPCB_API int mpcb_solve_held_windows_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                 const double *state, const double *v_beta, const double *target, const double *origin,
                                 const double *threshold, const uint8_t *flags,
                                 double *best_cost, int64_t *best_index, double *best_traj, double *first_control,
                                 int32_t *window_shape);
MPCB_API int mpcb_solve_held_windows_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N,
                                   const double *state, const double *v_beta, const double *target, const double *origin,
                                   const double *threshold, const uint8_t *flags,
                                   double *best_cost, int64_t *best_index, double *best_traj, double *first_control,
                                   int32_t *window_shape);

/* Closed loop of the FULL-tree scripts for a batch of robots (math_model.py:234-254 / run_math_model.py:261-276):
 * every tick solves all still-running robots in ONE batched FULL solve with the CARRIED threshold
 * (optimal_criterion is only lowered by an accepted leaf, math_model.py:195-198), applies the first pose of the
 * accepted path -- or repeats the previous one when nothing beats the threshold -- counts repeated positions
 * (stop at 2: "Recursive error") and tests is_on_target, all on the device; the host only reads one counter per tick.
 *   init_state[N][3], target[N][2], origin[N][2], first_threshold[N] (control_criterion of the start pose)
 *   out_log[N][max_ticks][5] = the 5-list each tick returns, out_ticks[N], out_status[N] (MPCB_LOOP_*) */
MPCB_API int mpcb_full_closed_loop_host(mpcb_handle *h, int cost_kind, int H, int64_t N, const double *init_state,
                               const double *target, const double *origin, const double *first_threshold,
                               double eps, int max_ticks, double *out_log, int32_t *out_ticks, int32_t *out_status);

/* ONE oversized FULL tree per solve, shared by the ranks of an NCCL communicator (one process per GPU): rank r of R
 * expands the first controls of its contiguous, balanced share of [0, S) -- so rank order is leaf-index order --
 * and reduces it to a (float64 cost, int64 index) record per solve; ONE collective on the data path, an ncclAllGather
 * of those 16-byte records over NVLink, gives every rank all R of them (with the branch-and-bound or the screened
 * pass 1 a second 8-byte all-gather shares the ranks' initial upper bounds before the descent, so that a rank whose
 * share holds no good leaf still prunes against the best bound known); a local kernel takes their lexicographic minimum and every
 * rank re-rolls the winner's trajectory itself (no broadcast).  The only coupling between the leaves of the
 * reference's tree is the running strict-'<' minimum (math_model.py:195-198); this is its multi-GPU form.
 * Collective call: every rank of the communicator must make it with the same arguments (N solves, same states);
 * every rank receives the same outputs, as mpcb_solve_batch_* would return them for the whole tree.  Indices are
 * global leaf indices.  comm is an ncclComm_t created on the handle's device (mpcb_nccl_comm_create). */
MPCB_API int mpcb_solve_tree_split_device(mpcb_handle *h, void *nccl_comm, int cost_kind, int H, int64_t N,
                                 const double *state, const double *target, const double *origin,
                                 const double *threshold,
                                 double *best_cost, int64_t *best_index, double *best_traj, double *first_control);
MPCB_API int mpcb_solve_tree_split_host(mpcb_handle *h, void *nccl_comm, int cost_kind, int H, int64_t N,
                               const double *state, const double *target, const double *origin,
                               const double *threshold,
                               double *best_cost, int64_t *best_index, double *best_traj, double *first_control);

/* The reconciliation step on its own: lexicographic (cost, index) minimum over the ranks of an NCCL communicator,
 * in place on 1-element device buffers -- one 16-byte all-gather and a local minimum (exact for float64 costs and
 * 63-bit indices).  Ranks without a leaf (index < 0) or with a NaN cost never win; if no rank holds a leaf the
 * result is index -1 with the smallest cost reported (NaN if every cost is NaN).  The scratch lives in the handle. */
MPCB_API int mpcb_allreduce_min(mpcb_handle *h, void *nccl_comm, double *cost_dev, int64_t *index_dev);
/* NCCL bootstrap helpers (id is 128 bytes, generated on rank 0 and distributed by the caller); the communicator
 * is created on the handle's device. */
MPCB_API int mpcb_nccl_unique_id(void *id128);
MPCB_API int mpcb_nccl_comm_create(mpcb_handle *h, int nranks, int rank, const void *id128, void **comm_out);
MPCB_API int mpcb_nccl_comm_destroy(void *comm);

#ifdef __cplusplus
}
#endif
#endif /* MPCB200_H */
