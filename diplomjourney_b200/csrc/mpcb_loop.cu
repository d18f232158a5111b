// mpcb_loop.cu -- device-resident closed loop of the online (HELD) controller: SURVEY 8f rows f1+f2.
//
// One CTA per robot runs the whole tick loop of math_mpc(..., isActual=False)
// (math_model_tree.py:542-579) without returning to the host:
//   per tick  windows   vector_of_velocities / vector_of_beta_angles      math_model_tree.py:239-256
//             solve     HELD predictive_control, slow-down override        math_model_tree.py:308-361
//             apply     finishing heuristic m, result pose, threshold reset math_model_tree.py:388-429
//             stop      is_on_target, repeated-position ("Recursive error") math_model_tree.py:48-52,559-563
//             events    new_target / turn_left / turn_right + slow_down     math_model_tree.py:118-226,564-569
//             noise     (actual run only) get_actual_velocity / _beta_angle math_model_tree.py:259-275,590-597
// Operator events come as a script {tick, kind, a, b} (the reference's demo: turn_right at tick 60, turn_left at 90,
// new_target at 110); thread 0 applies an event after the tick it names, to the robot's own pose, and the CTA
// reloads target, line and cost constants from shared memory.
// The "actual" run (math_mpc(..., True)) gives every robot its own numpy RandomState (key[624] + pos, mpcb_noise.cuh):
// the CTA keeps it in shared memory while it runs the robot, and thread 0 perturbs the applied (v, beta) after every
// tick, draw for draw as the reference does.  A robot may instead draw from numpy's Generator(PCG64) (mpcb_pcg64.cuh):
// its 6-word record lives in thread 0's registers while the CTA runs the robot -- no shared memory, no twist.  The
// generator kind is a template parameter, so the noise-free loop stays free of all of it.
// rng_seed_kernel / pcg64_seed_kernel build those generators on the device from numpy's seeds.
//
// A HELD tick is tiny (S <= 451 candidates x H steps), so the loop is latency-bound, not
// throughput-bound: everything is evaluated directly in float64 with the reference's formula and
// operation order -- no fp32 stage, no refinement -- and the batch dimension (robots) fills the GPU.
#include "mpcb_events.cuh"
#include "mpcb_noise.cuh"
#include "mpcb_pcg64.cuh"

#include <cmath>

namespace mpcb {

constexpr int kLoopThreads = 256;
constexpr int kMaxWin = 128;     // max candidates per axis of the acceleration window

__device__ __forceinline__ void lex_min_d(double &J, int &j, double oJ, int oj) {
    if (oj >= 0 && (j < 0 || oJ < J || (oJ == J && oj < j))) { J = oJ; j = oj; }
}

struct LoopCost {
    double xt, yt, ox, oy, A, B, xt_oy, yt_ox, norm, theta;    // x_t y_0, y_t x_0: added one at a time
    int kind;
    __device__ double operator()(double x, double y, double phi) const {
        double dx = xt - x, dy = yt - y;
        double d = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
        double dl;
        if (x == ox && y == oy) dl = 1000.0;
        else dl = fabs(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(A, x), -__dmul_rn(B, y)), xt_oy), -yt_ox)) / norm;
        double dl2 = __dmul_rn(dl, dl);
        if (kind == 0) {
            double ang = theta - phi;
            return __dadd_rn(__dadd_rn(__dmul_rn(10000.0, d), __dmul_rn(10.0, __dmul_rn(ang, ang))),
                             __dmul_rn(100.0, dl2));
        }
        return __dadd_rn(__dmul_rn(10000.0, d), __dmul_rn(10000.0, dl2));
    }
};

// H steps of control (v, tan beta) from (x, y, phi); optionally records the poses
__device__ __forceinline__ void loop_walk(const mpcb_loop_params &p, double v, double tb, double &x, double &y,
                                          double &phi, double *poses) {
    const double dphi = __dmul_rn(__dmul_rn(__ddiv_rn(v, p.L), tb), p.delta_t);
    for (int k = 0; k < p.H; ++k) {
        phi = __dadd_rn(phi, dphi);
        double sn, cs;
        sincos(phi, &sn, &cs);
        x = __dadd_rn(x, __dmul_rn(__dmul_rn(v, cs), p.delta_t));
        y = __dadd_rn(y, __dmul_rn(__dmul_rn(v, sn), p.delta_t));
        if (poses) { poses[3 * k] = x; poses[3 * k + 1] = y; poses[3 * k + 2] = phi; }
    }
}

// Acceleration windows around the current (v, beta) (vector_of_velocities / vector_of_beta_angles,
// math_model_tree.py:239-256): candidate i is  v + delta_v (i - half_v)  kept if 0 <= . < v_max, resp.
// beta + delta_beta (i - half_beta)  kept if |.| <= beta_limit -- the same float64 expressions, order preserved.
// Warp 0 builds the velocity window, warp 1 the angle window (ballot + prefix count compaction, 32 candidates per
// round); out[0] = nV, out[1] = nB, *vslow = max(min V, v_min) (the slow-down override, :312-316).
// Needs >= 64 threads; the caller synchronises the CTA afterwards.
__device__ __forceinline__ void build_windows(const mpcb_loop_params &p, double v, double beta, double *s_V,
                                              double *s_B, int *out, double *vslow) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp > 1) return;
    const int n = warp == 0 ? p.n_v : p.n_beta;
    double *dst = warp == 0 ? s_V : s_B;
    int count = 0;
    double vmin = INFINITY;
    for (int i0 = 0; i0 < n && count < kMaxWin; i0 += 32) {
        const int i = i0 + lane;
        double c = 0.0;
        bool keep = false;
        if (i < n) {
            if (warp == 0) {
                c = __dadd_rn(v, __dmul_rn(p.delta_v, (double)i - p.half_v));
                keep = !(c < 0.0) && c < p.v_max;
            } else {
                c = __dadd_rn(beta, __dmul_rn(p.delta_beta, (double)i - p.half_beta));
                keep = fabs(c) <= p.beta_limit;
            }
        }
        const unsigned mk = __ballot_sync(0xffffffffu, keep);
        const int slot = count + __popc(mk & ((1u << lane) - 1u));
        if (keep && slot < kMaxWin) { dst[slot] = c; vmin = fmin(vmin, c); }
        count = min(count + __popc(mk), kMaxWin);
    }
    if (warp == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) vmin = fmin(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
        if (lane == 0) { out[0] = count; *vslow = vmin > p.v_min ? vmin : p.v_min; }
    } else if (lane == 0) {
        out[1] = count;
    }
}

// HELD solve of one robot over the windows in shared memory: candidate c = iv*nB + ib holds (v, beta) for all H
// steps; block-wide lexicographic (cost, index) minimum, result valid on thread 0.  Contains one CTA barrier.
__device__ __forceinline__ void held_block_solve(const mpcb_loop_params &p, const LoopCost &cost, const double *s_V,
                                                 const double *s_tanB, int nV, int nB, bool slow, double vslow,
                                                 double x0, double y0, double phi0, double *s_J, int *s_j,
                                                 double &bJ, int &bj) {
    const int tid = threadIdx.x;
    const int S = nV * nB;
    bJ = INFINITY; bj = -1;
    for (int c = tid; c < S; c += kLoopThreads) {
        const int iv = c / nB, ib = c - iv * nB;
        const double v = slow ? vslow : s_V[iv];
        double x = x0, y = y0, phi = phi0;
        loop_walk(p, v, s_tanB[ib], x, y, phi, nullptr);
        lex_min_d(bJ, bj, cost(x, y, phi), c);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oJ = __shfl_xor_sync(0xffffffffu, bJ, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        lex_min_d(bJ, bj, oJ, oj);
    }
    // (s_J / s_j of the previous solve were consumed before the CTA barriers that every caller has between two solves)
    if ((tid & 31) == 0) { s_J[tid >> 5] = bJ; s_j[tid >> 5] = bj; }
    __syncthreads();
    if (tid == 0)
        for (int i = 1; i < kLoopThreads / 32; ++i) lex_min_d(bJ, bj, s_J[i], s_j[i]);
}

// the line constants and the heading reference of a loaded target and line origin, rounded as the reference rounds
// them (no FMA contraction of A^2 + B^2)
__device__ __forceinline__ void line_consts(LoopCost &cost) {
    cost.A = cost.yt - cost.oy; cost.B = cost.xt - cost.ox;
    cost.xt_oy = __dmul_rn(cost.xt, cost.oy); cost.yt_ox = __dmul_rn(cost.yt, cost.ox);
    cost.norm = sqrt(__dadd_rn(__dmul_rn(cost.A, cost.A), __dmul_rn(cost.B, cost.B)));
    cost.theta = atan(cost.xt / cost.yt);
}

__device__ __forceinline__ void load_cost(LoopCost &cost, const double *target, const double *origin, long long n,
                                          int kind) {
    // (also called with n = 0 on the CTA's shared copy {x_t, y_t}, {x_0, y_0} after an operator event)
    cost.xt = target[2 * n]; cost.yt = target[2 * n + 1];
    cost.ox = origin[2 * n]; cost.oy = origin[2 * n + 1];
    line_consts(cost);
    cost.kind = kind;
}

enum LoopGen { kGenNone = 0, kGenMt19937 = 1, kGenPcg64 = 2 };    // the actual run's generator kind

// kTrace: the per-tick trace is written (LoopArgs::trace_*, each still nullable).  A template parameter, so that the loop
// without a trace is the very code it was before the trace existed (a uniform runtime test cost it 1-2 % of its time).
template <int kGen, bool kTrace>
__global__ void __launch_bounds__(kLoopThreads) held_loop_kernel(const LoopArgs a) {
    __shared__ double s_V[kMaxWin], s_B[kMaxWin], s_tanB[kMaxWin];
    __shared__ double s_J[kLoopThreads / 32];
    __shared__ int s_j[kLoopThreads / 32];
    __shared__ double s_state[5];      // x, y, phi, v, beta fed to the next tick
    // nV, nB, slow flag, stop decided at the top of a tick, stop decided at its bottom.  The two stop flags are
    // separate words: each is rewritten only after every thread has passed at least two CTA barriers since reading it.
    __shared__ int s_ctl[5];
    __shared__ double s_vslow;
    // operator events: x_t, y_t, x_0, y_0 as thread 0 last set them, and how many events it has applied (a counter, not
    // a flag: every thread compares it with its own copy after the tick's last barrier, so it never has to be cleared)
    __shared__ double s_line[4];
    __shared__ int s_events;
    extern __shared__ unsigned s_mt[];  // MT19937: the running robot's generator, key[624] + pos (dynamic, kMtWords words)
    const mpcb_loop_params &p = a.p;
    const int tid = threadIdx.x;
    if (tid == 0) s_events = 0;
    int seen_events = 0;

    for (long long n = blockIdx.x; n < a.N; n += gridDim.x) {
        LoopCost cost;
        load_cost(cost, a.target, a.origin, n, p.cost_kind);
        // thread-0 state of the loop (math_mpc locals and the module globals it touches)
        double thr = a.first_threshold ? a.first_threshold[n] : INFINITY;
        int slow_steps = a.slow_steps ? a.slow_steps[n] : 0;
        int m = 0, ticks = 0, status = 2;
        bool recursive = false, have_traj = false;
        double opt[3 * MPCB_MAX_H], res_v = 0.0, res_beta = 0.0;
        double xprev = 0.0, yprev = 0.0;
        Pcg64 pcg;                                 // PCG64: the running robot's generator (thread 0)
        __syncthreads();                           // the previous robot's shared state has been consumed
        if (tid == 0) {
            for (int k = 0; k < 5; ++k) s_state[k] = a.init[5 * n + k];
            xprev = s_state[0]; yprev = s_state[1];
            if constexpr (kGen == kGenPcg64) pcg = pcg64_load(a.pcg_state + (size_t)n * kPcgWords);
        }
        if constexpr (kGen == kGenMt19937)
            for (int i = tid; i < kMtWords; i += kLoopThreads) s_mt[i] = a.rng_state[(size_t)n * kMtWords + i];
        __syncthreads();

        for (;;) {
            // ---- stop test (thread 0) + acceleration windows (warps 0 and 1)
            if (tid == 0) {
                const double dx = cost.xt - s_state[0], dy = cost.yt - s_state[1];
                int stop = 0;        // rounded as is_on_target rounds it (no FMA contraction)
                if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= p.eps) { stop = 1; status = 0; }
                else if (ticks >= p.max_ticks) { stop = 1; status = 2; }
                s_ctl[2] = slow_steps > 0; s_ctl[3] = stop;
            }
            build_windows(p, s_state[3], s_state[4], s_V, s_B, s_ctl, &s_vslow);
            __syncthreads();
            if (s_ctl[3]) break;
            const int nV = s_ctl[0], nB = s_ctl[1];
            const bool slow = s_ctl[2] != 0;
            for (int i = tid; i < nB; i += kLoopThreads) s_tanB[i] = tan(s_B[i]);
            __syncthreads();

            // ---- HELD solve
            const double x0 = s_state[0], y0 = s_state[1], phi0 = s_state[2];
            double bJ; int bj;
            held_block_solve(p, cost, s_V, s_tanB, nV, nB, slow, s_vslow, x0, y0, phi0, s_J, s_j, bJ, bj);

            // ---- apply (thread 0)
            if (tid == 0) {
                const bool accepted = bj >= 0 && bJ < thr;  // strict '<' (math_model_tree.py:351)
                if (accepted) {
                    const int iv = bj / nB, ib = bj - iv * nB;
                    res_v = slow ? s_vslow : s_V[iv];
                    res_beta = s_B[ib];
                    double x = x0, y = y0, phi = phi0;
                    loop_walk(p, res_v, s_tanB[ib], x, y, phi, opt);
                    have_traj = true;
                }
                slow_steps -= 1;
                int stop = 0;
                if (!have_traj) { stop = 1; status = 3; }   // reference: IndexError on the [[[0]]] placeholder
                else {
                    // finishing heuristic (math_model_tree.py:392-414)
                    int pick = 0;
                    const int last = 3 * (p.H - 1);
                    if (m == 2) pick = 2;
                    else if (m == 1) { pick = 1; m += 1; }
                    else {
                        const double ex = cost.xt - opt[last], ey = cost.yt - opt[last + 1];
                        if (__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)) <= p.eps) m += 1;
                    }
                    if (pick > p.H - 1) pick = p.H - 1;
                    const double rx = opt[3 * pick], ry = opt[3 * pick + 1], rphi = opt[3 * pick + 2];
                    thr = 9223372036854775807.0;            // sys.maxsize (math_model_tree.py:428)
                    // the applied (v, beta): the commanded ones, or in the actual run what the actuators make of them
                    // (math_model_tree.py:590-597) -- velocity drawn first, then beta, and before the stall stop
                    double av = res_v, ab = res_beta;
                    if constexpr (kGen == kGenMt19937) {
                        av = actual_velocity(res_v, s_mt);
                        ab = actual_beta(res_beta, s_mt);
                    } else if constexpr (kGen == kGenPcg64) {
                        av = actual_velocity(res_v, pcg);
                        ab = actual_beta(res_beta, pcg);
                    }
                    const size_t row = (size_t)n * p.max_ticks + ticks;
                    double *log = a.out_log + row * 5;
                    log[0] = rx; log[1] = ry; log[2] = rphi; log[3] = av; log[4] = ab;
                    // the trace: what the reference's tick logs besides the 5-list (predicted_trajectory_*, result_v /
                    // result_beta); opt and res_* still hold the previous tick's when this one accepted no leaf
                    if constexpr (kTrace) {
                        if (a.trace_pred)
                            for (int k = 0; k < 3 * p.H; ++k) a.trace_pred[row * 3 * p.H + k] = opt[k];
                        if (a.trace_ctl) { a.trace_ctl[2 * row] = res_v; a.trace_ctl[2 * row + 1] = res_beta; }
                        if (a.trace_cost) a.trace_cost[row] = accepted ? bJ : NAN;
                    }
                    s_state[0] = rx; s_state[1] = ry; s_state[2] = rphi; s_state[3] = av; s_state[4] = ab;
                    ticks += 1;
                    if (recursive) { stop = 1; status = 1; }        // "Recursive error." (math_model_tree.py:559-561)
                    else {
                        if (rx == xprev && ry == yprev) recursive = true;
                        // operator events of this tick (math_model_tree.py:564-569), in script order
                        bool fired = false;
                        for (int e = 0; e < a.n_events; ++e)
                            if (a.events[e].tick == ticks) {
                                if (!fired) { s_line[0] = cost.xt; s_line[1] = cost.yt; s_line[2] = cost.ox; s_line[3] = cost.oy; }
                                apply_event(a.events[e], a.radius_u_turn, rx, ry, rphi, s_line, slow_steps);
                                fired = true;
                            }
                        if (fired) s_events += 1;
                    }
                    xprev = rx; yprev = ry;
                }
                s_ctl[4] = stop;
            }
            __syncthreads();
            if (s_ctl[4]) break;
            if (s_events != seen_events) {          // uniform: written before the barrier above
                seen_events = s_events;
                load_cost(cost, s_line, s_line + 2, 0, p.cost_kind);
            }
        }
        if (tid == 0) {
            a.out_ticks[n] = ticks;
            a.out_status[n] = status;
            if (a.out_final) {
                double *f = a.out_final + 6 * n;
                f[0] = cost.xt; f[1] = cost.yt; f[2] = cost.ox; f[3] = cost.oy; f[4] = (double)slow_steps; f[5] = (double)m;
            }
            if constexpr (kGen == kGenPcg64) pcg64_store(pcg, a.pcg_state + (size_t)n * kPcgWords);
        }
        if constexpr (kGen == kGenMt19937)       // thread 0's last draw came before the barrier that ended the loop
            for (int i = tid; i < kMtWords; i += kLoopThreads) a.rng_state[(size_t)n * kMtWords + i] = s_mt[i];
    }
}

// The generators of the actual run, seeded as numpy's RandomState(keys[n]) (key_len == 0) or RandomState(keys[n, :])
// (keys[N][key_len]): one thread per generator writes its [625] record straight to global memory -- the recurrences
// are serial, so there is nothing to split inside a generator.
__global__ void __launch_bounds__(128) rng_seed_kernel(long long N, const unsigned *keys, int key_len, unsigned *rng_state) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= N) return;
    unsigned *st = rng_state + (size_t)n * kMtWords;
    if (key_len == 0) mt_seed(st, keys[n]);
    else mt_seed_by_array(st, keys + (size_t)n * key_len, key_len);
}

cudaError_t launch_rng_seed(cudaStream_t st, long long N, const unsigned *keys, int key_len, unsigned *rng_state) {
    rng_seed_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(N, keys, key_len, rng_state);
    return cudaGetLastError();
}

// The Generator(PCG64) records of the actual run, seeded as default_rng(SeedSequence(entropy, spawn_key)): one thread per
// generator hashes its words into the 4-word pool and writes its [6] record.  entropy[ent_len] is shared by all
// generators (ent_stride 0) or one row per generator (ent_stride = ent_len); spawn[N][spawn_len] (spawn_len 0: none).
__global__ void __launch_bounds__(128) pcg64_seed_kernel(long long N, const unsigned *entropy, int ent_len,
                                                         int ent_stride, const unsigned *spawn, int spawn_len,
                                                         unsigned long long *pcg_state) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= N) return;
    pcg64_seed(entropy + (size_t)n * ent_stride, ent_len, spawn ? spawn + (size_t)n * spawn_len : nullptr, spawn_len,
               pcg_state + (size_t)n * kPcgWords);
}

cudaError_t launch_pcg64_seed(cudaStream_t st, long long N, const unsigned *entropy, int ent_len, int ent_stride,
                              const unsigned *spawn, int spawn_len, unsigned long long *pcg_state) {
    pcg64_seed_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(N, entropy, ent_len, ent_stride, spawn, spawn_len,
                                                                   pcg_state);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// ONE online tick for a batch of robots that each have their OWN acceleration window (SURVEY 8f row f2): the window
// is rebuilt per robot and per tick around the robot's current (v, beta) (math_model_tree.py:239-256, called at
// :543-545 and, with the noisy actuator values, at :590-597), so a batch of robots shares no grid.  One CTA per
// robot: windows on the device, HELD solve in float64 with the reference's formula, the winner re-rolled -- one
// launch for the whole batch.  index = iv * nB + ib within the robot's own window (shape returned).
__global__ void __launch_bounds__(kLoopThreads) held_windows_kernel(const WindowArgs a) {
    __shared__ double s_V[kMaxWin], s_B[kMaxWin], s_tanB[kMaxWin];
    __shared__ double s_J[kLoopThreads / 32];
    __shared__ int s_j[kLoopThreads / 32];
    __shared__ int s_n[2];
    __shared__ double s_vslow;
    const mpcb_loop_params &p = a.p;
    const int tid = threadIdx.x;
    for (long long n = blockIdx.x; n < a.N; n += gridDim.x) {
        const int fl = a.flags ? (int)a.flags[n] : 0;
        double *traj = a.out_traj ? a.out_traj + (size_t)n * 3 * p.H : nullptr;
        auto none = [&](int nV, int nB) {              // no candidate / entry not to be solved
            if (a.out_cost) a.out_cost[n] = NAN;
            if (a.out_index) a.out_index[n] = -1;
            if (traj) for (int k = 0; k < 3 * p.H; ++k) traj[k] = NAN;
            if (a.out_ctl) { a.out_ctl[2 * n] = NAN; a.out_ctl[2 * n + 1] = NAN; }
            if (a.out_shape) { a.out_shape[2 * n] = nV; a.out_shape[2 * n + 1] = nB; }
        };
        if (fl & MPCB_FLAG_SKIP) { if (tid == 0) none(0, 0); continue; }
        LoopCost cost;
        load_cost(cost, a.target, a.origin, n, p.cost_kind);
        __syncthreads();                           // the previous robot's windows have been consumed
        build_windows(p, a.vbeta[2 * n], a.vbeta[2 * n + 1], s_V, s_B, s_n, &s_vslow);
        __syncthreads();
        const int nV = s_n[0], nB = s_n[1];
        for (int i = tid; i < nB; i += kLoopThreads) s_tanB[i] = tan(s_B[i]);
        __syncthreads();
        const bool slow = (fl & MPCB_FLAG_SLOW) != 0;
        const double x0 = a.state[3 * n], y0 = a.state[3 * n + 1], phi0 = a.state[3 * n + 2];
        double bJ; int bj;
        held_block_solve(p, cost, s_V, s_tanB, nV, nB, slow, s_vslow, x0, y0, phi0, s_J, s_j, bJ, bj);
        if (tid == 0) {
            if (bj < 0) { none(nV, nB); continue; }
            const double thr = a.threshold ? a.threshold[n] : INFINITY;
            const int iv = bj / nB, ib = bj - iv * nB;
            const double v = slow ? s_vslow : s_V[iv];
            double x = x0, y = y0, phi = phi0, tr[3 * MPCB_MAX_H];
            loop_walk(p, v, s_tanB[ib], x, y, phi, tr);
            if (traj) for (int k = 0; k < 3 * p.H; ++k) traj[k] = tr[k];
            if (a.out_cost) a.out_cost[n] = bJ;
            if (a.out_index) a.out_index[n] = bJ < thr ? bj : -1;       // strict '<' (math_model_tree.py:351)
            if (a.out_ctl) { a.out_ctl[2 * n] = v; a.out_ctl[2 * n + 1] = s_B[ib]; }
            if (a.out_shape) { a.out_shape[2 * n] = nV; a.out_shape[2 * n + 1] = nB; }
        }
    }
}

cudaError_t launch_held_windows(cudaStream_t st, const WindowArgs &a, int sms) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, held_windows_kernel, kLoopThreads, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    long long grid = (long long)sms * per_sm;
    if (grid > a.N) grid = a.N;
    held_windows_kernel<<<(unsigned)grid, kLoopThreads, 0, st>>>(a);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// One HELD solve per CTA straight from the raw grids (v[nv], beta[nb]) in float64: the low-latency
// path of the per-tick host API (S <= a few thousand candidates; no tables, no fp32 stage, one launch).
__global__ void __launch_bounds__(kLoopThreads) held_small_kernel(const SmallArgs a) {
    extern __shared__ double s_tan[];
    __shared__ double s_J[kLoopThreads / 32];
    __shared__ int s_j[kLoopThreads / 32];
    const int tid = threadIdx.x;
    const long long n = blockIdx.x;
    mpcb_loop_params p{};
    p.L = a.L; p.delta_t = a.delta_t; p.H = a.H;
    LoopCost cost;
    cost.xt = a.target[2 * n]; cost.yt = a.target[2 * n + 1];
    cost.ox = a.origin[2 * n]; cost.oy = a.origin[2 * n + 1];
    line_consts(cost);
    cost.kind = a.cost_kind;
    const int fl = a.flags ? (int)a.flags[n] : 0;
    const bool slow = (fl & MPCB_FLAG_SLOW) != 0;
    if (fl & MPCB_FLAG_SKIP) {                      // entry of a batch that is not to be solved
        if (tid == 0) {
            a.out_cost[n] = NAN; a.out_index[n] = -1;
            for (int k = 0; k < 3 * a.H; ++k) a.out_traj[(size_t)n * 3 * a.H + k] = NAN;
            a.out_ctl[2 * n] = NAN; a.out_ctl[2 * n + 1] = NAN;
        }
        return;
    }
    for (int i = tid; i < a.nb; i += kLoopThreads) s_tan[i] = tan(a.beta[i]);
    __syncthreads();
    const double x0 = a.state[3 * n], y0 = a.state[3 * n + 1], phi0 = a.state[3 * n + 2];
    const int S = a.nv * a.nb;
    double bJ = INFINITY; int bj = -1;
    for (int c = tid; c < S; c += kLoopThreads) {
        const int iv = c / a.nb, ib = c - iv * a.nb;
        const double v = slow ? a.v_slow : a.v[iv];
        double x = x0, y = y0, phi = phi0;
        loop_walk(p, v, s_tan[ib], x, y, phi, nullptr);
        lex_min_d(bJ, bj, cost(x, y, phi), c);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oJ = __shfl_xor_sync(0xffffffffu, bJ, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        lex_min_d(bJ, bj, oJ, oj);
    }
    if ((tid & 31) == 0) { s_J[tid >> 5] = bJ; s_j[tid >> 5] = bj; }
    __syncthreads();
    if (tid == 0) {
        for (int i = 1; i < kLoopThreads / 32; ++i) lex_min_d(bJ, bj, s_J[i], s_j[i]);
        const double thr = a.threshold ? a.threshold[n] : INFINITY;
        double *traj = a.out_traj + (size_t)n * 3 * a.H;
        if (bj >= 0) {
            const int iv = bj / a.nb, ib = bj - iv * a.nb;
            const double v = slow ? a.v_slow : a.v[iv];
            double x = x0, y = y0, phi = phi0;
            loop_walk(p, v, s_tan[ib], x, y, phi, traj);
            a.out_cost[n] = bJ;
            a.out_index[n] = bJ < thr ? bj : -1;
            a.out_ctl[2 * n] = v; a.out_ctl[2 * n + 1] = a.beta[ib];
        } else {
            a.out_cost[n] = NAN; a.out_index[n] = -1;
            for (int k = 0; k < 3 * a.H; ++k) traj[k] = NAN;
            a.out_ctl[2 * n] = NAN; a.out_ctl[2 * n + 1] = NAN;
        }
    }
}

cudaError_t launch_held_small(cudaStream_t st, const SmallArgs &a) {
    held_small_kernel<<<(unsigned)a.N, kLoopThreads, sizeof(double) * a.nb, st>>>(a);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// FULL closed loop, one graph launch (mpcb_api.cu, full_loop_enqueue):
//   init -> gate -> WHILE (running > 0 && tick < max_ticks) { batched solve; apply; gate }
// The running count is ctl[0] (FullLoopArgs::active_count), the tick ctl[1] (FullLoopArgs::tick); both are zero when
// the init kernel runs, and the gate zeroes the count after reading it, for the apply kernel of the next tick.

// What the loop does before tick 0, one thread per robot: the robot's state and threshold (+inf without first_threshold),
// zeroed counters, and the on-target test of math_model.py:239 -- a robot on target at entry never runs.
__global__ void full_loop_init_kernel(const FullLoopArgs a, const double *init, const double *first_threshold) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    const double x = init[3 * n], y = init[3 * n + 1];
    a.state[3 * n] = x; a.state[3 * n + 1] = y; a.state[3 * n + 2] = init[3 * n + 2];
    a.threshold[n] = first_threshold ? first_threshold[n] : INFINITY;
    a.kcount[n] = 0; a.have_ret[n] = 0; a.ticks[n] = 0;
    // rounded as is_on_target rounds it (no FMA contraction): a robot on the boundary starts as the reference's does
    const double dx = a.target[2 * n] - x, dy = a.target[2 * n + 1] - y;
    const bool on_target = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= a.eps;
    a.status[n] = on_target ? MPCB_LOOP_ON_TARGET : -1;
    a.flags[n] = on_target ? MPCB_FLAG_SKIP : 0;
    if (!on_target) atomicAdd(a.active_count, 1);
}

// The WHILE node's condition (one thread): advance the tick (advance = 0 ahead of the loop, 1 at the end of a tick) and
// take the running count, leaving it zero.
__global__ void full_loop_gate_kernel(cudaGraphConditionalHandle cond, int *ctl, int max_ticks, int advance) {
    const int tick = ctl[1] + advance, running = ctl[0];
    ctl[0] = 0;
    ctl[1] = tick;
    cudaGraphSetConditional(cond, running > 0 && tick < max_ticks ? 1u : 0u);
}

cudaError_t launch_full_loop_init(cudaStream_t st, const FullLoopArgs &a, const double *init, const double *first_threshold) {
    const int bs = 128;
    full_loop_init_kernel<<<(unsigned)((a.N + bs - 1) / bs), bs, 0, st>>>(a, init, first_threshold);
    return cudaGetLastError();
}

cudaError_t launch_full_loop_gate(cudaStream_t st, cudaGraphConditionalHandle cond, int *ctl, int max_ticks, int advance) {
    full_loop_gate_kernel<<<1, 1, 0, st>>>(cond, ctl, max_ticks, advance);
    return cudaGetLastError();
}

// What the host loop of math_model.py:239-254 does between two predictive_control calls, one thread per robot, after
// the tick's batched solve.
__global__ void full_apply_kernel(const FullLoopArgs a) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N || a.status[n] >= 0) return;
    const int tick = *a.tick;
    double ret[5];
    const long long idx = a.best_index[n];
    const double *tr = a.best_traj + (size_t)n * 3 * a.H;
    if (idx >= 0) {                                        // a leaf beat the carried optimum (strict '<')
        ret[0] = tr[0]; ret[1] = tr[1]; ret[2] = tr[2];
        ret[3] = a.first_control[2 * n]; ret[4] = a.first_control[2 * n + 1];
        a.threshold[n] = a.best_cost[n];
        a.have_ret[n] = 1;
    } else if (!a.have_ret[n]) {                           // reference: IndexError on the placeholder trajectory
        a.status[n] = MPCB_LOOP_NO_LEAF;
        a.flags[n] = MPCB_FLAG_SKIP;
        return;
    } else {                                               // stall: the previous path is returned again
        for (int k = 0; k < 5; ++k) ret[k] = a.last_ret[5 * n + k];
    }
    const size_t row = (size_t)n * a.max_ticks + tick;
    double *log = a.log + row * 5;
    for (int k = 0; k < 5; ++k) { log[k] = ret[k]; a.last_ret[5 * n + k] = ret[k]; }
    if (a.trace_pred) {                                    // a stall repeats the last accepted trajectory
        double *last = a.last_traj + (size_t)n * 3 * a.H;
        for (int k = 0; k < 3 * a.H; ++k) {
            if (idx >= 0) last[k] = tr[k];
            a.trace_pred[row * 3 * a.H + k] = last[k];
        }
    }
    if (a.trace_ctl) { a.trace_ctl[2 * row] = ret[3]; a.trace_ctl[2 * row + 1] = ret[4]; }
    if (a.trace_cost) a.trace_cost[row] = idx >= 0 ? a.best_cost[n] : NAN;
    const double xprev = a.state[3 * n], yprev = a.state[3 * n + 1];
    a.state[3 * n] = ret[0]; a.state[3 * n + 1] = ret[1]; a.state[3 * n + 2] = ret[2];
    a.ticks[n] = tick + 1;
    int k = a.kcount[n];
    if (ret[0] == xprev && ret[1] == yprev) a.kcount[n] = ++k;
    const double dx = a.target[2 * n] - ret[0], dy = a.target[2 * n + 1] - ret[1];
    int status = -1;
    if (k == 2) status = MPCB_LOOP_STALLED;
    else if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= a.eps) status = MPCB_LOOP_ON_TARGET;   // as is_on_target
    else if (tick + 1 >= a.max_ticks) status = MPCB_LOOP_MAX_TICKS;
    if (status >= 0) { a.status[n] = status; a.flags[n] = MPCB_FLAG_SKIP; }
    else atomicAdd(a.active_count, 1);
}

cudaError_t launch_full_apply(cudaStream_t st, const FullLoopArgs &a) {
    const int bs = 128;
    full_apply_kernel<<<(unsigned)((a.N + bs - 1) / bs), bs, 0, st>>>(a);
    return cudaGetLastError();
}

template <int kGen, bool kTrace>
static cudaError_t launch_held_loop_t(cudaStream_t st, const LoopArgs &a, int sms) {
    const size_t smem = kGen == kGenMt19937 ? sizeof(unsigned) * kMtWords : 0;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, held_loop_kernel<kGen, kTrace>, kLoopThreads, smem) !=
            cudaSuccess || per_sm < 1)
        per_sm = 1;
    long long grid = (long long)sms * per_sm;
    if (grid > a.N) grid = a.N;
    held_loop_kernel<kGen, kTrace><<<(unsigned)grid, kLoopThreads, smem, st>>>(a);
    return cudaGetLastError();
}

template <bool kTrace>
static cudaError_t launch_held_loop_gen(cudaStream_t st, const LoopArgs &a, int sms) {
    if (a.rng_state) return launch_held_loop_t<kGenMt19937, kTrace>(st, a, sms);
    if (a.pcg_state) return launch_held_loop_t<kGenPcg64, kTrace>(st, a, sms);
    return launch_held_loop_t<kGenNone, kTrace>(st, a, sms);
}

cudaError_t launch_held_loop(cudaStream_t st, const LoopArgs &a, int sms) {
    if (a.trace_pred || a.trace_ctl || a.trace_cost) return launch_held_loop_gen<true>(st, a, sms);
    return launch_held_loop_gen<false>(st, a, sms);
}

}  // namespace mpcb
