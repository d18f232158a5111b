// mpcb_types.cuh -- device-side data layout shared by the kernels and the host API.
//
// Everything a kernel needs lives in three places:
//   GridTables   per control grid, built once by mpcb_set_grid (read-only, L2/L1 resident)
//   SolveParams  one 272-byte record per MPC solve, built on the device by prep_kernel
//   LaunchArgs   per launch, passed by value (constant bank)
#pragma once
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/mpcb200.h"
#include "mpcb_screen.cuh"

namespace mpcb {

#ifndef MPCB_THREADS
#define MPCB_THREADS 256
#endif
constexpr int kThreads = MPCB_THREADS;   // threads per CTA; one "unit" (leaf or depth-(H-1) node) per thread
constexpr int kPrefixCta = 1024;   // pass 1 of the prefix kernel runs ONE 1024-thread CTA per SM (measured +4-6 % over
                                   // 4 x 256); it covers four 256-node tiles at a time, so segments, the refinement
                                   // pass and the work list keep their 256-node granularity
constexpr int kMaxH = 8;
constexpr int kLeafChunk = 1024;   // float4 entries of the per-control leaf table staged in shared memory

// cost weights (math_model.py:86 / math_model_tree.py:87)
constexpr double kWd = 10000.0;

#ifdef __CUDACC__
#define MPCB_HD __host__ __device__ __forceinline__
#define MPCB_HD_NOINLINE __host__ __device__ __noinline__
#else
#define MPCB_HD inline
#define MPCB_HD_NOINLINE inline
#endif

// round-to-nearest add / mul / sqrt that the compiler must not contract into FMAs (the reference evaluates
// x + v*cos(phi)*dt as separate operations), and a read-only load
MPCB_HD double dadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
MPCB_HD double dmul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
MPCB_HD double dsqrt(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return std::sqrt(a);
#endif
}
MPCB_HD double ro_load(const double *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// Division of a 64-bit index by an invariant divisor (Granlund-Montgomery round-up form).  Host/device: the CPU
// test-suite checks the very same code (tests/test_shipped_code_on_host.py).
struct FastDiv64 {
    unsigned long long m;   // magic
    unsigned long long d;   // divisor
    unsigned sh1, sh2;
    MPCB_HD unsigned long long div(unsigned long long n) const {
#ifdef __CUDA_ARCH__
        unsigned long long t = __umul64hi(m, n);
#else
        unsigned long long t = (unsigned long long)(((unsigned __int128)m * n) >> 64);
#endif
        return (t + ((n - t) >> sh1)) >> sh2;
    }
};

// 32-bit flavour (indices below 2^32): 5 instructions per quotient instead of ~15
struct FastDiv32 {
    unsigned m, d, sh1, sh2;
    MPCB_HD unsigned div(unsigned n) const {
#ifdef __CUDA_ARCH__
        unsigned t = __umulhi(m, n);
#else
        unsigned t = (unsigned)(((unsigned long long)m * n) >> 32);
#endif
        return (t + ((n - t) >> sh1)) >> sh2;
    }
};

inline void fastdiv32_init(FastDiv32 &f, unsigned long long d64) {
    unsigned d = (unsigned)d64;
    f.d = d;
    if (d <= 1) { f.m = 0; f.sh1 = 0; f.sh2 = 0; return; }
    unsigned l = 0;
    while ((l < 32) && ((1ULL << l) < d)) ++l;
    f.m = (unsigned)((((1ULL << l) - d) << 32) / d) + 1u;
    f.sh1 = 1; f.sh2 = l - 1;
}

inline void fastdiv_init(FastDiv64 &f, unsigned long long d) {
    f.d = d;
    if (d <= 1) { f.m = 0; f.sh1 = 0; f.sh2 = 0; return; }
    unsigned l = 0;
    while ((l < 64) && ((1ULL << l) < d)) ++l;            // ceil(log2 d), d < 2^63
    unsigned __int128 num = ((unsigned __int128)1 << 64) * (((unsigned __int128)1 << l) - d);
    f.m = (unsigned long long)(num / d) + 1ULL;
    f.sh1 = 1; f.sh2 = l - 1;
}

constexpr int kLeafPerThread = 8;  // leafwalk: leaves per thread per tile (tile = kThreads * kLeafPerThread leaves)

// Per control grid. c = iv*nb + ib.
struct GridTables {
    // float64, for the depth-(H-1) prefix walk and the exact re-evaluation
    const double4 *tab64;       // {cos dphi_c, sin dphi_c, s_c = v_c*dt, dphi_c}
    const double  *vtab;        // v_c
    const float4  *tab32;       // tab64 rounded to float: the walk of the fp32 pre-filter (pruned pass 1)
    const double4 *tab64_slow;  // same with every v := max(min V, v_min)   (math_model_tree.py:312-316)
    const double  *vtab_slow;
    const double  *beta;        // beta[nb]
    // float32, for the inner loops
    const float4 *leaf32;       // {a_c = s_c cos dphi_c, b_c = s_c sin dphi_c, r_c = s_c^2, g_c = sqrt(10) dphi_c}
    const float4 *leaf32p;      // pair table: [2m] = {a_2m, a_2m+1, b_2m, b_2m+1}, [2m+1] = {r.., r.., g.., g..}; odd S pads by repeating the last leaf
    const float4 *leaf32r;      // the pair table laid out by SPEED ROW (row iv = ppr pairs of its nb leaves, an odd row padded by
                                // repeating its last leaf): all leaves of a row share r_c = (v dt)^2; null when it does not fit one chunk
    int nv, ppr;                // speeds; pairs per row = (nb + 1) / 2
    const float2 *ctl32;        // {dphi_c, s_c}
    const float2 *ctl32_slow;
    int S, nb;
    double dt;
    double smax, dphimax;       // max |s_c|, max |dphi_c| (both variants) -- error model, pruning bounds
    double smin;                // min s_c (both variants) -- pruning bounds
    ScreenBox sbox;             // range of leaf32's a, b, g: the intervals of stage 1 of the two-stage screen (mpcb_screen.cuh)
};

// The {a_2m, a_2m+1, b_2m, b_2m+1} half of the row table (GridTables::leaf32r), for the stage-1 loop of the two-stage
// screen, which reads it through the uniform datapath.  Filled by mpcb_set_grid when the row table exists and passed
// BY VALUE to the exhaustive pass-1 kernel (a __grid_constant__ parameter), so every launch carries its own handle's
// table: handles with different grids may solve concurrently on one device.  A row table fits one shared-memory chunk
// (2 nv ppr <= kLeafChunk float4), so kLeafChunk / 2 pairs hold every one of them: 8 KiB of the 32,764 bytes a kernel's
// parameters may take.
constexpr int kRowPairCap = kLeafChunk / 2;
struct RowPairs { float4 ab[kRowPairCap]; };

// Per solve (float64). Built by prep_kernel from the raw inputs.
struct __align__(16) SolveParams {
    double xs, ys, phi0;        // start pose
    double xt, yt;              // target
    double ox, oy;              // origin of the tracked line
    double theta;               // arctan(x_t / y_t)                         (math_model.py:83)
    double lineA, lineB, lineC, line_norm;   // (y_t-y_0), (x_t-x_0), x_t y_0 - y_t x_0, sqrt(A^2+B^2)
                                // (lineC only forms the anchor e0: a leaf's line distance adds x_t y_0 and y_t x_0 one at
                                // a time, as the reference does -- one precomputed difference rounds otherwise far from (0, 0))
    double threshold;
    // start-frame quantities (frame: origin at the start position, x axis along the start heading)
    double u0, w0, d0;          // target, distance to target
    double e0, nx0, ny0;        // wl * signed line distance of the start, and its gradient
    double hp0;                 // wh * (theta - phi0)
    double wl, wh;              // sqrt of the line / heading weights
    double inv_wl;              // 1 / wl (the bounds normalise the line gradient by it)
    double Kbase;               // kWd d0 + e0^2 + hp0^2 (cost terms of the start pose): J = Kbase + J_rel
    double tol;                 // 2 x error bound of the fp32 leaf value that pass 2 filters with (leaf_val / leafwalk)
    double tol1;                // 2 x error bound of the value pass 1 RANKS with (prefix: direct form; else = tol)
    double special;             // 1e6 * wl^2: squared line term of the "on the origin" special case
    int flags;                  // bit0 slow, bit1 start_is_origin, bit2 near (leafwalk regime)
    int pad;
    // the start-frame quantities rounded to float once per solve, for the fp32 pre-filter of the pruned passes
    // (mpcb_bounds.cuh: prefilter_solve_consts / prefilter32): u0, w0, d0, e0, nx0, ny0, hp0, wl, 1/wl, wh
    float pf[12];
};
constexpr int kFlagSlow = 1, kFlagStartIsOrigin = 2, kFlagNear = 4, kFlagSkip = 8;

// refinement: a leaf whose fp32 value lies inside the window, waiting for its float64 evaluation (pass 2 lists them,
// cand_eval_kernel evaluates them one thread each)
struct __align__(8) Candidate { long long j; double jrel; int n; int pad; };

// refinement: a depth-(H-1) node whose bound reaches into the window, with the fp32 registers its leaves are scored
// from (refine_prefix_kernel lists them, refine_scan_kernel scans each with one warp)
struct __align__(16) RefineNode {
    float u, w, u2, w2, D2, Dp, nu, nw, e2, h2;   // ParentRegs of the form pass 2 filters with
    float thr, Lspecial;                          // window edge relative to the node, value of the special-case leaves
    double base;
    unsigned long long p;                         // node index
    int n;                                        // solve; -1 = slot reserved but not filled (list overflow)
    unsigned flags;                               // bit0 near, bit1 special
};

struct LaunchArgs {
    GridTables g;
    const SolveParams *sp;
    FastDiv64 fd[kMaxH];        // fd[k].d = S^(H-1-k)
    FastDiv32 fd32[kMaxH];      // same divisors, valid when idx32 != 0 (every index and divisor < 2^32); [1..] also when node32 != 0
    FastDiv64 fd_tiles, fd_S;   // division by tiles_per_solve and by S (the pruned kernels decode a global tile number per tile)
    int idx32;
    int node32;                 // prefix algorithm: every depth-(H-1) node index < 2^32 -> node_digits decodes with fd32
    unsigned step_digits[kMaxH]; // base-S digits of kThreads (most significant first): leafwalk advances a leaf index by kThreads
    int lw_smem;                // leafwalk FULL: stage ctl32 in shared memory (S <= 4096)
    unsigned tile_units;        // units per tile: kThreads (prefix) or kThreads*kLeafPerThread (leafwalk)
    int mode, H, cost_kind, refine;
    long long N;
    unsigned long long u_begin, u_end;     // unit range of every solve (leaves or depth-(H-1) nodes)
    unsigned long long tiles_per_solve, segs_per_solve, total_segs;
    unsigned tps;                          // tiles per segment
    double *segmin;                        // [total_segs]  pass-1 partial minima of J_rel
    // refinement
    const unsigned *worklist;              // qualifying segment ids
    const unsigned *work_count;
    double *bestJ;                         // [N] exact cost of the best candidate so far
    long long *bestIdx;                    // [N]
    int *lock;                             // [N]
    unsigned long long *counters;          // [0] refine segments, [1] candidates, [2] pruned depth-(H-1) nodes, [3] same, frontier descent (added to [2] when the descent completes),
                                           // [7] nodes that passed stage 1 of the two-stage screen ([4..6] are other fields of the same buffer)
    unsigned long long *ub;                // [N] ordered key of an upper bound on each solve's minimal J_rel (pruning), or null
    int prune;
    int prefilter;                         // pruned pass 1: fp32 pre-filter of the node bound (mpcb_bounds.cuh)
    int screen;                            // exhaustive prefix pass 1: 0 = MUFU.SQRT per leaf, 1 = screened (sqrt only on nodes that can matter),
                                           // 2 = screened in two stages (distance first, mpcb_screen.cuh)
    float bc32[7];                         // smax, smin, dphimax, cosk[0], sink[0], cosk[1], sink[1] rounded to float (fp32 pre-filter)
    double cosk[kMaxH], sink[kMaxH];       // cos / sin of (i+1) dphi_max: the heading range reachable in i+1 steps (cos = -2: the whole circle)
    // subtree cut (pruned pass 1, H >= 3): tiles that survived the depth-(H-2) bound, as global tile numbers
    // n * tiles_per_solve + tile; null = walk every tile
    const unsigned long long *tile_list;
    const unsigned *tile_count;
    // frontier descent (pruned pass 1, H >= 3): surviving depth-(H-2) nodes as global ids n * S^(H-2) + index;
    // pass 1 then walks their children.  q_overflow != 0: a frontier outgrew its list -> the tile path takes over.
    const unsigned long long *q_list;
    const unsigned *q_count;
    unsigned q_cap;
    const unsigned *q_overflow;
    int gate;                              // 1: pass 1 returns at once if *q_overflow (frontier mode)
    int dump_direct;                       // prefix dump: direct (pass-1) form instead of the pass-2 form
    int npt;                               // depth-(H-1) nodes per thread in the exhaustive prefix pass 1 (1 or 2)
    int i0_begin, i0_end;                   // first-control range of this launch (probe)
    const double *tau;                     // [N] J_rel window upper edge
    // candidate list of the refinement (null: every candidate is evaluated where it is found)
    unsigned long long *refine_ctr;        // next work item of the refinement filter (handed out dynamically)
    RefineNode *node_list; unsigned *node_count; unsigned node_cap;    // null / 0: nodes are scanned where they are found
    Candidate *cand; unsigned *cand_count; unsigned cand_cap;
    double *cand_J;                        // [cand_cap] float64 cost of each listed candidate
    unsigned long long *cand_key;          // [N] ordered key of the smallest listed cost per solve
    unsigned long long *cand_idx;          // [N] smallest leaf index among the listed candidates of that cost
    // dump
    float4 *dump;                          // {x, y, phi, J_rel} per leaf
    unsigned long long dump_begin, dump_count;
};

// split tree: one rank's (cost, index) record of one solve -- what the ranks all-gather (mpcb_nccl.cu)
struct __align__(16) SplitRec { double cost; long long index; };

// device-resident closed loop (mpcb_loop.cu)
struct LoopArgs {
    mpcb_loop_params p;
    long long N;
    const double *init, *target, *origin, *first_threshold;
    const int *slow_steps;
    double *out_log;
    int *out_ticks, *out_status;
    // operator events applied between ticks (device copies; n_events = 0: none)
    const mpcb_loop_event *events;
    int n_events;
    double radius_u_turn;
    double *out_final;                                 // [N][6] x_t, y_t, x_0, y_0, steps_for_slowing, m; nullable
    unsigned *rng_state;                               // [N][625] numpy MT19937 key + pos, updated in place; null: no noise
    unsigned long long *pcg_state;                     // [N][6] numpy PCG64 records, updated in place (with rng_state null)
    // per-tick trace, written on out_log's row (nullable): optimal_trajectory's poses [N][max_ticks][H][3], the commanded
    // (v, beta) before actuator noise [N][max_ticks][2], the accepted leaf's cost [N][max_ticks] (NaN: none accepted)
    double *trace_pred, *trace_ctl, *trace_cost;
};

// one step of the online controller on per-robot records (mpcb_loop.cu, held_ctrl_step_kernel); all pointers are device
struct HeldCtrlArgs {
    mpcb_loop_params p;
    long long N;
    mpcb_held_ctrl *ctrl;                              // [N] in/out
    const double *measured;                            // [N][5] applied state of the pending proposals, nullable
    const mpcb_loop_event *events;                     // [N][n_ev], nullable with n_ev == 0
    int n_ev;
    double radius_u_turn;
    double *proposal;                                  // [N][5], nullable
    int *running;                                      // robots holding a proposal after the step (added), nullable
};

// one online tick of a batch of robots with per-robot acceleration windows (mpcb_loop.cu); all pointers are device
struct WindowArgs {
    mpcb_loop_params p;
    long long N;
    const double *state, *vbeta, *target, *origin, *threshold;   // [N][3], [N][2] (current v, beta), [N][2], [N][2], [N] or null
    const unsigned char *flags;                                   // MPCB_FLAG_* per robot, nullable
    double *out_cost; long long *out_index; double *out_traj, *out_ctl;
    int *out_shape;                                               // [N][2] = (nV, nB) of each robot's window, nullable
};

// per-tick bookkeeping of the FULL closed loop (mpcb_loop.cu)
struct FullLoopArgs {
    long long N;
    int H, max_ticks;
    const int *tick;                                   // the tick being applied (device counter, advanced by the gate)
    double eps;
    const double *target;                              // [N][2]
    const double *best_cost; const long long *best_index; const double *best_traj, *first_control;   // this tick's solve
    double *state, *threshold, *last_ret;              // [N][3], [N], [N][5]
    int *kcount, *have_ret, *status, *ticks;           // [N]
    unsigned char *flags;                              // [N] MPCB_FLAG_SKIP once a robot has stopped
    double *log;                                       // [N][max_ticks][5]
    int *active_count;                                 // robots still running after this tick
    double *trace_pred, *trace_ctl, *trace_cost;       // per-tick trace as in LoopArgs (nullable)
    double *last_traj;                                 // [N][H][3] the last accepted trajectory (needed with trace_pred)
};

// one-launch float64 HELD solve from the raw grids (mpcb_loop.cu); all pointers are device
struct SmallArgs {
    const double *v, *beta;            // raw grids
    const double *state, *target, *origin, *threshold, *flags;   // flags: MPCB_FLAG_* bits stored as doubles, nullable
    double *out_cost; long long *out_index; double *out_traj, *out_ctl;
    double L, delta_t, v_slow;
    int nv, nb, H, cost_kind;
    long long N;
};

}  // namespace mpcb
