// mpcb_kernels.cu -- sm_100a kernels of the MPC inner loop.
//
// Reference semantics implemented here (paths into ShittyWizard/DiplomJourney):
//   node step   iteration_of_predict          math_model.py:110-114
//   cost        control_criterion             math_model.py:82-86 (MM), math_model_tree.py:82-87 (TREE)
//   FULL tree   predictive_control            math_model.py:159-200
//   HELD tree   predictive_control            math_model_tree.py:308-361, CoordinateTree.py:20-30
//
// Numerical scheme (DESIGN.md section 3): every leaf cost is evaluated in fp32 as an OFFSET
// from a float64 anchor, J = Kbase + base_p + L, where L is O(reach) instead of O(1e5); a
// first pass keeps only partial minima, a second pass re-evaluates in float64 (reference
// formula, reference operation order) the few leaves whose fp32 value lies inside a
// rigorous error window above the minimum, so the selected leaf is the float64 argmin.
//
// Two expansion algorithms:
//   leafwalk  one thread per leaf walks all H steps in registers (sin.approx/cos.approx)
//   prefix    one thread per depth-(H-1) node: float64 walk of the shared prefix, then a
//             loop over the S children with the per-control displacement table in shared
//             memory (no MUFU sin/cos in the inner loop: the child pose is a rotation of a
//             tabulated displacement into the parent frame)
// Pass 1 of either only RANKS (cheaper "direct" forms under their own error bound tol1, leaf_val_direct /
// leaf_walk_direct); pass 2 filters with the accurate offset form before the float64 re-evaluation.
//
// Exact branch-and-bound (option prune, DESIGN.md section 3.5): lower bounds on the cost of every leaf below a
// node (projection_range, lower_bound_from, subtree_lower_bound) against a running upper bound cut nodes in pass 1, 256-node
// tiles before pass 1 (tilecut_kernel) or whole subtrees from the root down (frontier_expand_kernel); the
// records returned are bit-identical to evaluating every leaf.
#include <type_traits>

#include "mpcb_types.cuh"
#include "mpcb_bounds.cuh"   // walk_step, projection_range, lower_bound_from, subtree_lower_bound (host/device)
#include "mpcb_exact.cuh"    // exact_step, exact_terminal, exact_cost (host/device)

#ifndef MPCB_UNROLL2
#define MPCB_UNROLL2 8  // pairs per unrolled iteration of the two-node loop (4: -3.5 %, profiles/r1j_variants.txt)
#endif
#ifndef MPCB_UNROLL4
#define MPCB_UNROLL4 2  // pairs per unrolled iteration of the four-node loop (1, 2, 4 within 1.3 %)
#endif
#ifndef MPCB_PN_CTA2
#define MPCB_PN_CTA2 512  // threads per CTA of the two-nodes-per-thread pass-1 kernel (one CTA per SM, four 256-node tiles per
                          // work item).  Row loop (the usual case): 384 / 512 / 640 threads = 3.13 / 3.20 / 3.14e12 rollouts/s on the
                          // cfg2 bench; flat screen loop: 512 / 640 / 768 / 896 / 1024 = 2.99 / 3.10 / 2.96 / 2.98 / 2.97e12
                          // (profiles/r2c_variants.txt, r2f_variants.txt, r2u_variants.txt, r2v_variants.txt)
#endif
#ifndef MPCB_UNROLL_ROWS
#define MPCB_UNROLL_ROWS 4  // pairs per unrolled iteration of the row loop (a row of the cfg2 grid has 21 pairs: 3 / 4 / 7 / 8 / 21
                            // = 3.15 / 3.20 / 3.20 / 3.07 / 3.17e12)
#endif
#ifndef MPCB_UNROLL_DIST
#define MPCB_UNROLL_DIST 7  // pairs per unrolled iteration of the stage-1 row loop of the two-stage screen (a cfg2 row = 3 x 7 pairs)
#endif
#ifndef MPCB_UNROLL
#define MPCB_UNROLL 8   // pairs per unrolled iteration of the pass-1 loop (4..16 are within 1 %, profiles/r1b_variants.txt)
#endif

#include <cfloat>
#include <cmath>

namespace mpcb {

// ------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ float sqrt_approx(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ double4 ldg_d4(const double4 *p) {
    const double2 *q = reinterpret_cast<const double2 *>(p);
    double2 a = __ldg(q), b = __ldg(q + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// order-preserving map double -> uint64 (non-NaN), so that partial minima can be folded with
// atomicMin; ~0 is the "nothing yet" value the host memsets
__device__ __forceinline__ unsigned long long ordered_key(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return b ^ ((b >> 63) ? ~0ULL : 0x8000000000000000ULL);
}
__device__ __forceinline__ double ordered_value(unsigned long long k) {
    if (k == ~0ULL) return INFINITY;
    unsigned long long b = (k >> 63) ? (k ^ 0x8000000000000000ULL) : ~k;
    return __longlong_as_double((long long)b);
}
// lexicographic (cost, index) minimum; NaN costs never win
__device__ __forceinline__ void lex_min(double &J, long long &j, double oJ, long long oj) {
    if (oj >= 0 && (j < 0 || oJ < J || (oJ == J && oj < j))) { J = oJ; j = oj; }
}

// The quantities one "parent" (the start pose for leafwalk, a depth-(H-1) node for prefix)
// contributes to the cost of its leaves, in the parent's own frame.
struct ParentRegs {
    float u, w;        // target in the parent frame
    float u2, w2;      // -2u, -2w
    float D2, Dp;      // |target|^2, |target|
    float nu, nw;      // wl * unit normal of the tracked line, parent frame
    float e2, h2;      // 2 * wl*signed line distance of the parent, 2 * wh*(theta - phi_parent)
    float eh, nhh;     // direct form (prefix pass 1): e2/2, -h2/2
    float u2s, w2s, D2s; // direct form: kWd^2 * (-2u, -2w, |target|^2), so that sqrt() returns kWd * d
                         // (leafwalk, whose leaves are not one table step away: u2s, w2s = kWd * (u, w) instead)
};

// fp32 leaf part L of the cost: J_leaf = Kbase + base_parent + L,
//   L = 1e4 (d - Dp) + line offset + heading offset.
//   (a, b) displacement parent->leaf in the parent frame, r = a^2+b^2, g = wh * heading change
//   FAR  (|target| >= 4 reach): d - Dp = num / (d + Dp), num = r - 2(u a + w b): no cancellation
//   NEAR: d - Dp = |(u - a, w - b)| - float(Dp); the float64 remainder of Dp sits in the base
template <bool HEAD, bool NEAR>
__device__ __forceinline__ float leaf_val(float a, float b, float r, float g, const ParentRegs &p) {
    float t;
    if (NEAR) {
        float dx = p.u - a, dy = p.w - b;
        t = sqrt_approx(__fmaf_rn(dx, dx, dy * dy)) - p.Dp;
    } else {
        float num = __fmaf_rn(p.u2, a, __fmaf_rn(p.w2, b, r));
        float d = sqrt_approx(p.D2 + num);
        t = num * rcp_approx(d + p.Dp);
    }
    float q = __fmaf_rn(p.nu, a, p.nw * b);
    float acc = q * (p.e2 + q);
    if (HEAD) acc = __fmaf_rn(g, g - p.h2, acc);
    return __fmaf_rn(10000.0f, t, acc);
}

// DIRECT form of the same leaf part (prefix pass 1, FAR regime), 8 FP32 ops + 1 MUFU per leaf instead of 14 + 1.5:
//   L' = sqrt(kWd^2 (D2 + num)) + (q + eh)^2 + (g + nhh)^2,   eh = e2/2, nhh = -h2/2
// i.e. L' = L + kWd Dp + eh^2 + nhh^2 in exact arithmetic: the weight kWd sits under the root (the node's u2, w2, D2
// are scaled by kWd^2 in float64 before rounding, the table's r by one FFMA), and the node constant is taken out of
// the minimum altogether -- parent_setup's base_direct subtracts it in float64.  The value is therefore rounded at
// the magnitude of kWd d (not of kWd reach), so this form only RANKS leaves for pass 1 with its own, wider error
// bound tol1 (prep_kernel); pass 2 filters with leaf_val.
constexpr float kWd2f = 1.0e8f;          // kWd^2, exact in fp32
template <bool HEAD>
__device__ __forceinline__ float leaf_val_direct(float a, float b, float r, float g, const ParentRegs &p) {
    const float dd = __fmaf_rn(p.u2s, a, __fmaf_rn(p.w2s, b, __fmaf_rn(kWd2f, r, p.D2s)));
    const float s = sqrt_approx(dd);
    const float q = __fmaf_rn(p.nu, a, __fmaf_rn(p.nw, b, p.eh));
    float acc = __fmaf_rn(q, q, s);
    if (HEAD) { const float gg = g + p.nhh; acc = __fmaf_rn(gg, gg, acc); }
    return acc;
}

// returns the remainder term -kWd (Dp - float(Dp)) that a NEAR parent adds to its base
__device__ __forceinline__ double split_distance(double Dp, ParentRegs &pr) {
    pr.D2 = (float)(Dp * Dp);
    pr.Dp = (float)Dp;
    return -kWd * (Dp - (double)pr.Dp);
}

// the start pose as the "parent" of every leaf (leafwalk); returns its base (remainder term only)
__device__ __forceinline__ double start_as_parent(const SolveParams &P, ParentRegs &pr) {
    pr.u = (float)P.u0; pr.w = (float)P.w0;
    pr.u2 = (float)(-2.0 * P.u0); pr.w2 = (float)(-2.0 * P.w0);
    const double rem = split_distance(P.d0, pr);
    const double base = (P.flags & kFlagNear) ? rem : 0.0;
    pr.nu = (float)P.nx0; pr.nw = (float)P.ny0;
    pr.e2 = (float)(2.0 * P.e0); pr.h2 = (float)(2.0 * P.hp0);
    // direct form (pass 1): leaf_walk_direct
    pr.u2s = (float)(kWd * P.u0); pr.w2s = (float)(kWd * P.w0);
    pr.eh = (float)P.e0; pr.nhh = (float)(-P.hp0);
    return base;
}

// what the direct form of the leafwalk measures from: L' = L + kWd d0 + eh^2 + nhh^2 (see leaf_walk_direct)
__device__ __forceinline__ double start_direct_offset(const SolveParams &P, const ParentRegs &pr) {
    return kWd * P.d0 + (double)pr.eh * (double)pr.eh + (double)pr.nhh * (double)pr.nhh;
}

// DIRECT form for a leaf reached by a walk (leafwalk pass 1): (xi, eta, psi) is the leaf in the start frame,
//   L' = kWd |(u, w) - (xi, eta)| + (q + e0)^2 + (wh psi - hp0)^2,
// 9 FP32 ops + 1 MUFU against 15 + 2 for leaf_val, and no FAR/NEAR distinction.  Like leaf_val_direct it is rounded at
// the magnitude of kWd d and only RANKS (tol1); pass 2 filters with leaf_val.
template <bool HEAD>
__device__ __forceinline__ float leaf_walk_direct(float xi, float eta, float psi, const ParentRegs &p) {
    const float dx = __fmaf_rn(-10000.0f, xi, p.u2s), dy = __fmaf_rn(-10000.0f, eta, p.w2s);
    const float s = sqrt_approx(__fmaf_rn(dx, dx, dy * dy));
    const float q = __fmaf_rn(p.nu, xi, __fmaf_rn(p.nw, eta, p.eh));
    float acc = __fmaf_rn(q, q, s);
    if (HEAD) { const float gg = __fmaf_rn(3.16227766016837952f, psi, p.nhh); acc = __fmaf_rn(gg, gg, acc); }
    return acc;
}

// A depth-(H-1) node in float64: its pose from the walk of its prefix (i_0 .. i_{H-2}) in the start frame, and the
// quantities of its own frame that its children's costs (and the bound over them) are built from.
struct NodeFrame {
    double u, w, Dp;           // target in the node's frame, its distance
    double ep, nu, nw;         // scaled line distance of the node, gradient of the scaled line distance in the node's frame
    double hp;                 // scaled heading error
    double base0;              // J_rel of the node's own terms: kWd (Dp - d0) + (ep^2 - e0^2) + (hp^2 - hp0^2)
    bool unmoved;              // the node has not moved at all (the reference's "on the line origin" special case)
};

__device__ __forceinline__ void node_frame(const LaunchArgs &a, const SolveParams &P, unsigned long long p, NodeFrame &f) {
    double xi = 0.0, eta = 0.0, psi = 0.0, cp = 1.0, sp = 0.0;
    node_digits(a, p, [&](unsigned i) { walk_step(ldg_d4(a.g.tab64 + i), xi, eta, psi, cp, sp); });
    f.unmoved = (xi == 0.0 && eta == 0.0);
    const double relx = P.u0 - xi, rely = P.w0 - eta;
    f.u = cp * relx + sp * rely; f.w = cp * rely - sp * relx;
    f.Dp = sqrt(f.u * f.u + f.w * f.w);
    f.ep = P.e0 + P.nx0 * xi + P.ny0 * eta;
    f.nu = cp * P.nx0 + sp * P.ny0; f.nw = cp * P.ny0 - sp * P.nx0;
    f.hp = P.hp0 - P.wh * psi;
    // J_rel is measured from the start pose's own cost terms: Kbase = kWd d0 + e0^2 + hp0^2
    f.base0 = kWd * (f.Dp - P.d0) + (f.ep - P.e0) * (f.ep + P.e0) + (f.hp - P.hp0) * (f.hp + P.hp0);
}

// fp32 pre-filter (mpcb_bounds.cuh): true = the float64 bound over the children of node p exceeds `bound` for certain
// (the float bound from a float walk exceeds it by more than 8 tol1), so the node need not be set up in float64 at all
__device__ __forceinline__ bool node_far32(const LaunchArgs &a, const SolveParams &P, unsigned long long p, double bound) {
    const Prefilter32 pf = prefilter32(a, P);
    float xi = 0.f, eta = 0.f, psi = 0.f, cp = 1.f, sp = 0.f;
    node_digits(a, p, [&](unsigned i) {
        const float4 t = __ldg(a.g.tab32 + i);
        walk_step_t<float>(t.x, t.y, t.z, t.w, xi, eta, psi, cp, sp);
    });
    return node_prefilter32(pf, xi, eta, psi, cp, sp) > __double2float_ru(bound + 8.0 * P.tol1);
}

// no child can do better than: one step as straight at the target as the steering allows, the most favourable line offset
// that step can produce and the most favourable heading offset (lower_bound_from); in the node's own frame the heading
// is (1, 0), the target (u, w), the line gradient (nu, nw)
__device__ __forceinline__ double node_lower_bound(const LaunchArgs &a, const SolveParams &P, const NodeFrame &f) {
    return lower_bound_from(a, P, f.u, f.w, f.Dp, f.nu, f.nw, 1.0, 0.0, f.ep, f.hp, f.base0, 1);
}

// the fp32 registers of a node that survived (the conversions are only paid for nodes whose children are scored);
// returns base_p (with the remainder term of a NEAR node) and, for the direct form, base_direct
__device__ __forceinline__ double node_regs(const LaunchArgs &a, const NodeFrame &f, ParentRegs &pr, bool &near,
                                            double *base_direct) {
    pr.u = (float)f.u; pr.w = (float)f.w;
    pr.u2 = (float)(-2.0 * f.u); pr.w2 = (float)(-2.0 * f.w);
    const double dp_rem = split_distance(f.Dp, pr);
    pr.nu = (float)f.nu; pr.nw = (float)f.nw;
    pr.e2 = (float)(2.0 * f.ep); pr.h2 = (float)(2.0 * f.hp);
    near = !(f.Dp >= 4.0 * a.g.smax);
    if (base_direct) {
        pr.eh = 0.5f * pr.e2; pr.nhh = -0.5f * pr.h2;
        pr.u2s = (float)(-2.0 * kWd * kWd * f.u); pr.w2s = (float)(-2.0 * kWd * kWd * f.w);
        pr.D2s = (float)(kWd * kWd * (f.Dp * f.Dp));
        *base_direct = f.base0 - kWd * f.Dp - (double)pr.eh * (double)pr.eh - (double)pr.nhh * (double)pr.nhh;
    }
    return f.base0 + (near ? dp_rem : 0.0);
}

// all of it at once.  Returns base_p (float64) and whether the node has not moved at all.
__device__ __forceinline__ double parent_setup(const LaunchArgs &a, const SolveParams &P,
                                               unsigned long long p, ParentRegs &pr, bool &near, bool &unmoved,
                                               double *lower_bound = nullptr, double *base_direct = nullptr) {
    NodeFrame f;
    node_frame(a, P, p, f);
    unmoved = f.unmoved;
    if (lower_bound) *lower_bound = node_lower_bound(a, P, f);
    return node_regs(a, f, pr, near, base_direct);
}

// candidate found by the refinement filter: listed for cand_eval_kernel (float64 evaluation, one thread per candidate:
// the in-window leaves of a solve cluster in a few nodes, and a thread evaluating its node's candidates one after the
// other -- three double-precision sincos each -- was most of pass 2); true = listed
__device__ __forceinline__ bool cand_push(const LaunchArgs &a, long long n, long long j, double jrel) {
    if (!a.cand) return false;
    const unsigned slot = atomicAdd(a.cand_count, 1u);
    if (slot >= a.cand_cap) return false;                  // list full: the caller evaluates it where it stands
    Candidate c;
    c.j = j; c.jrel = jrel; c.n = (int)n; c.pad = 0;
    a.cand[slot] = c;
    return true;
}

// ... or, when the list is full, evaluated on the spot and folded into the thread's running best
__device__ __forceinline__ void take_candidate(const LaunchArgs &a, const SolveParams &P, long long n, long long j,
                                               double jrel32, double &bJ, long long &bj) {
    atomicAdd(a.counters + 1, 1ULL);
    if (cand_push(a, n, j, jrel32)) return;
    double J = a.refine ? exact_cost(a, P, j, nullptr, nullptr) : (P.Kbase + jrel32);
    lex_min(bJ, bj, J, j);
}

// block-wide lexicographic min, then one locked update of the solve's record
__device__ __forceinline__ void publish_best(const LaunchArgs &a, long long n, double bJ, long long bj,
                                             double *s_J, long long *s_j) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double oJ = __shfl_xor_sync(0xffffffffu, bJ, o);
        long long oj = __shfl_xor_sync(0xffffffffu, bj, o);
        lex_min(bJ, bj, oJ, oj);
    }
    if (lane == 0) { s_J[warp] = bJ; s_j[warp] = bj; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < kThreads / 32; ++i) lex_min(bJ, bj, s_J[i], s_j[i]);
        if (bj >= 0) {
            while (atomicCAS(a.lock + n, 0, 1) != 0) {}
            __threadfence();
            double cJ = *(volatile double *)(a.bestJ + n);
            long long cj = *(volatile long long *)(a.bestIdx + n);
            lex_min(cJ, cj, bJ, bj);
            *(volatile double *)(a.bestJ + n) = cJ;
            *(volatile long long *)(a.bestIdx + n) = cj;
            __threadfence();
            atomicExch(a.lock + n, 0);
        }
    }
    __syncthreads();
}

// pass 1: every warp folds its partial minimum into the segment's key -- no CTA barrier.  Under the screen almost every
// node publishes INFINITY, so a warp without a finite value skips the reduction (it would publish nothing anyway).
__device__ __forceinline__ void publish_segmin(const LaunchArgs &a, unsigned seg, double v) {
    if (!__any_sync(0xffffffffu, v < INFINITY)) return;
    v = warp_min(v);
    if ((threadIdx.x & 31) == 0 && v < INFINITY)
        atomicMin(reinterpret_cast<unsigned long long *>(a.segmin) + seg, ordered_key(v));
}

// the same when the lanes of a warp may belong to different segments (frontier mode: a warp's 32 nodes can straddle
// a 256-node tile boundary when S is not a multiple of 32)
__device__ __forceinline__ void publish_segmin_lanes(const LaunchArgs &a, unsigned seg, double v) {
    const unsigned live = __ballot_sync(0xffffffffu, v < INFINITY);
    if (!live) return;
    const unsigned seg0 = __shfl_sync(0xffffffffu, seg, __ffs(live) - 1);
    if (__all_sync(0xffffffffu, !(v < INFINITY) || seg == seg0)) publish_segmin(a, seg0, v);
    else if (v < INFINITY) atomicMin(reinterpret_cast<unsigned long long *>(a.segmin) + seg, ordered_key(v));
}

// frontier mode: pass 1 must not walk a list that a frontier outgrew (the host then redoes it through the tile bound)
__device__ __forceinline__ bool gate_closed(const LaunchArgs &a) {
    return a.gate != 0 && *(volatile const unsigned *)a.q_overflow != 0;
}

// work item -> (segment, solve, tile range).  PASS 1 walks all segments, PASS 2 the work list.
template <int PASS>
__device__ __forceinline__ void decode_work(const LaunchArgs &a, unsigned long long w, unsigned &seg,
                                            long long &n, unsigned long long &tile_lo, unsigned long long &tile_hi) {
    const unsigned sps = (unsigned)a.segs_per_solve;
    unsigned long long off;
    if (PASS == 1) { seg = (unsigned)w; off = 0; }
    else {
        unsigned long long e = a.tps == 1 ? w : w / a.tps;
        seg = a.worklist[e];
        off = w - e * a.tps;
    }
    unsigned nn = seg / sps;
    unsigned sidx = seg - nn * sps;
    n = nn;
    tile_lo = (unsigned long long)sidx * a.tps + off;
    tile_hi = tile_lo + (PASS == 1 ? a.tps : 1);
    if (tile_hi > a.tiles_per_solve) tile_hi = a.tiles_per_solve;
}

// ------------------------------------------------------------------------------------ prefix
// One thread per depth-(H-1) node; the S children are scored from the shared-memory table.
// Pass-1 inner loops over the PAIR table: entry m holds leaves 2m, 2m+1 as
//   tab[2m] = {a0, a1, b0, b1}, tab[2m+1] = {r0, r1, g0, g1}
// so that two leaves go through one packed FFMA2/FADD2/FMUL2 each (sm_100 f32x2 pipe): the
// FP32 part costs half the issue slots and the loop becomes XU(MUFU)-bound.
template <bool HEAD>
__device__ __forceinline__ float prefix_min_loop_far2(const float4 *__restrict__ tab, int npairs, const ParentRegs &pr,
                                                      float best) {
    const float2 U2 = make_float2(pr.u2s, pr.u2s), W2 = make_float2(pr.w2s, pr.w2s);
    const float2 D2 = make_float2(pr.D2s, pr.D2s), K2 = make_float2(kWd2f, kWd2f);
    const float2 NU = make_float2(pr.nu, pr.nu), NW = make_float2(pr.nw, pr.nw);
    const float2 EH = make_float2(pr.eh, pr.eh), NHH = make_float2(pr.nhh, pr.nhh);
    constexpr int kUnroll = MPCB_UNROLL;
#pragma unroll kUnroll
    for (int m = 0; m < npairs; ++m) {
        const float4 t0 = tab[2 * m], t1 = tab[2 * m + 1];
        const float2 A = make_float2(t0.x, t0.y), B = make_float2(t0.z, t0.w);
        const float2 R = make_float2(t1.x, t1.y), G = make_float2(t1.z, t1.w);
        // leaf_val_direct on two leaves at a time
        const float2 dd = __ffma2_rn(U2, A, __ffma2_rn(W2, B, __ffma2_rn(K2, R, D2)));
        const float2 q = __ffma2_rn(NU, A, __ffma2_rn(NW, B, EH));
        float2 acc = __ffma2_rn(q, q, make_float2(sqrt_approx(dd.x), sqrt_approx(dd.y)));
        if (HEAD) { const float2 gg = __fadd2_rn(G, NHH); acc = __ffma2_rn(gg, gg, acc); }
        best = fminf(best, fminf(acc.x, acc.y));
    }
    return best;
}

// The same loop for ONE node shared by the warp (pruned pass 1, sparse survivors): lane l scores leaf pairs l, l + 32,
// ...; the caller reduces over the lanes.  Per leaf the arithmetic is that of prefix_min_loop_far2 and the minimum does
// not depend on the order it is taken in, so the node's value is bit-identical.
template <bool HEAD>
__device__ __forceinline__ float prefix_min_loop_far2_lanes(const float4 *__restrict__ tab, int npairs, float u2s, float w2s,
                                                            float D2s, float nu, float nw, float eh, float nhh, int lane) {
    const float2 U2 = make_float2(u2s, u2s), W2 = make_float2(w2s, w2s), D2 = make_float2(D2s, D2s);
    const float2 K2 = make_float2(kWd2f, kWd2f), NU = make_float2(nu, nu), NW = make_float2(nw, nw);
    const float2 EH = make_float2(eh, eh), NHH = make_float2(nhh, nhh);
    float best = INFINITY;
    for (int m = lane; m < npairs; m += 32) {
        const float4 t0 = tab[2 * m], t1 = tab[2 * m + 1];
        const float2 A = make_float2(t0.x, t0.y), B = make_float2(t0.z, t0.w);
        const float2 R = make_float2(t1.x, t1.y), G = make_float2(t1.z, t1.w);
        const float2 dd = __ffma2_rn(U2, A, __ffma2_rn(W2, B, __ffma2_rn(K2, R, D2)));
        const float2 q = __ffma2_rn(NU, A, __ffma2_rn(NW, B, EH));
        float2 acc = __ffma2_rn(q, q, make_float2(sqrt_approx(dd.x), sqrt_approx(dd.y)));
        if (HEAD) { const float2 gg = __fadd2_rn(G, NHH); acc = __ffma2_rn(gg, gg, acc); }
        best = fminf(best, fminf(acc.x, acc.y));
    }
    return best;
}

// NPT depth-(H-1) nodes per thread on the same table entry: the two LDS.128 of a leaf pair feed all of the thread's nodes
template <bool HEAD, int NPT>
__device__ __forceinline__ void prefix_min_loop_far2xN(const float4 *__restrict__ tab, int npairs,
                                                       const ParentRegs (&p)[NPT], float (&best)[NPT]) {
    float2 U[NPT], W[NPT], D[NPT], NU[NPT], NW[NPT], E[NPT], Hh[NPT];
    float b[NPT];
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
        U[k] = make_float2(p[k].u2s, p[k].u2s); W[k] = make_float2(p[k].w2s, p[k].w2s);
        D[k] = make_float2(p[k].D2s, p[k].D2s);
        NU[k] = make_float2(p[k].nu, p[k].nu); NW[k] = make_float2(p[k].nw, p[k].nw);
        E[k] = make_float2(p[k].eh, p[k].eh); Hh[k] = make_float2(p[k].nhh, p[k].nhh);
        b[k] = best[k];
    }
    const float2 K2 = make_float2(kWd2f, kWd2f);
    constexpr int kUnroll = NPT == 2 ? MPCB_UNROLL2 : MPCB_UNROLL4;
#pragma unroll kUnroll
    for (int m = 0; m < npairs; ++m) {
        const float4 t0 = tab[2 * m], t1 = tab[2 * m + 1];
        const float2 A = make_float2(t0.x, t0.y), B = make_float2(t0.z, t0.w);
        const float2 R = make_float2(t1.x, t1.y), G = make_float2(t1.z, t1.w);
#pragma unroll
        for (int k = 0; k < NPT; ++k) {
            const float2 dd = __ffma2_rn(U[k], A, __ffma2_rn(W[k], B, __ffma2_rn(K2, R, D[k])));
            const float2 q = __ffma2_rn(NU[k], A, __ffma2_rn(NW[k], B, E[k]));
            float2 acc = __ffma2_rn(q, q, make_float2(sqrt_approx(dd.x), sqrt_approx(dd.y)));
            if (HEAD) { const float2 gg = __fadd2_rn(G, Hh[k]); acc = __ffma2_rn(gg, gg, acc); }
            b[k] = fminf(b[k], fminf(acc.x, acc.y));
        }
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) best[k] = b[k];
}

// SCREENED flavour of the same loop (option "screen", the default of the exhaustive pass 1): every leaf's cost terms are
// formed exactly as in leaf_val_direct -- dd (scaled squared distance to the target), q (line offset), gg (heading
// offset) -- but the MUFU.SQRT that turns them into the value L' = sqrt(dd) + q^2 + gg^2 is only spent on nodes that
// hold a leaf which can still matter.  With cn an upper bound (in the node's direct-form units, error margins
// included) on the value of any leaf that could be the solve's minimum,
//      L' < cn   <=>   sqrt(dd) < t,  t = cn - q^2 - gg^2   <=>   t > 0 and t^2 - dd > 0,
// and fma(t, t, -dd) is correctly rounded, so its sign is that of t^2 - dd for the fp32 t and dd at hand.  The loop
// keeps the maximum of t^2 - dd over the node's leaves: 9 packed FP32 ops + 1 FMNMX3 per node and leaf pair and no
// MUFU (against 8 + 2 MUFU.SQRT + 1).  A node whose maximum is positive is re-run through prefix_min_loop_far2 (the
// values it then publishes are the ones the unscreened kernel publishes); t < 0 with t^2 > dd is a harmless false hit.
template <bool HEAD, int NPT>
__device__ __forceinline__ void prefix_screen_loop_far2xN(const float4 *__restrict__ tab, int npairs,
                                                          const ParentRegs (&p)[NPT], const float (&cn)[NPT],
                                                          float (&mx)[NPT]) {
    float2 U[NPT], W[NPT], D[NPT], NU[NPT], NW[NPT], E[NPT], Hh[NPT], C[NPT];
    float m[NPT];
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
        // negated, so that the last FFMA2 forms t^2 - dd directly
        U[k] = make_float2(-p[k].u2s, -p[k].u2s); W[k] = make_float2(-p[k].w2s, -p[k].w2s);
        D[k] = make_float2(-p[k].D2s, -p[k].D2s);
        NU[k] = make_float2(p[k].nu, p[k].nu); NW[k] = make_float2(p[k].nw, p[k].nw);
        E[k] = make_float2(p[k].eh, p[k].eh); Hh[k] = make_float2(p[k].nhh, p[k].nhh);
        C[k] = make_float2(cn[k], cn[k]);
        m[k] = -INFINITY;
    }
    const float2 K2 = make_float2(-kWd2f, -kWd2f);
    constexpr int kUnroll = NPT == 2 ? MPCB_UNROLL2 : MPCB_UNROLL4;
#pragma unroll kUnroll
    for (int i = 0; i < npairs; ++i) {
        const float4 t0 = tab[2 * i], t1 = tab[2 * i + 1];
        const float2 A = make_float2(t0.x, t0.y), B = make_float2(t0.z, t0.w);
        const float2 R = make_float2(t1.x, t1.y), G = make_float2(t1.z, t1.w);
#pragma unroll
        for (int k = 0; k < NPT; ++k) {
            const float2 ndd = __ffma2_rn(U[k], A, __ffma2_rn(W[k], B, __ffma2_rn(K2, R, D[k])));      // -dd
            const float2 q = __ffma2_rn(NU[k], A, __ffma2_rn(NW[k], B, E[k]));
            float2 t = __ffma2_rn(make_float2(-q.x, -q.y), q, C[k]);
            if (HEAD) { const float2 gg = __fadd2_rn(G, Hh[k]); t = __ffma2_rn(make_float2(-gg.x, -gg.y), gg, t); }
            const float2 df = __ffma2_rn(t, t, ndd);
            m[k] = fmaxf(m[k], fmaxf(df.x, df.y));
        }
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) mx[k] = m[k];
}

// The screen loop over the ROW table (GridTables::leaf32r): all leaves of a speed row share r_c = (v dt)^2, so the
// innermost term of dd, fma(kWd^2, r, D2s), is formed once per node and row instead of once per pair -- 7 FFMA2 + 1 FADD2
// per node and leaf pair instead of 8 + 1, and the very same value (same operands, same operation).  The pairs an odd
// row is padded with repeat its last leaf, which changes no maximum.
template <bool HEAD, int NPT>
__device__ __forceinline__ void prefix_screen_loop_rows(const float4 *__restrict__ tab, int nv, int ppr,
                                                        const ParentRegs (&p)[NPT], const float (&cn)[NPT],
                                                        float (&mx)[NPT]) {
    float2 U[NPT], W[NPT], NU[NPT], NW[NPT], E[NPT], Hh[NPT], C[NPT];
    float nD[NPT], m[NPT];
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
        U[k] = make_float2(-p[k].u2s, -p[k].u2s); W[k] = make_float2(-p[k].w2s, -p[k].w2s);
        nD[k] = -p[k].D2s;
        NU[k] = make_float2(p[k].nu, p[k].nu); NW[k] = make_float2(p[k].nw, p[k].nw);
        E[k] = make_float2(p[k].eh, p[k].eh); Hh[k] = make_float2(p[k].nhh, p[k].nhh);
        C[k] = make_float2(cn[k], cn[k]);
        m[k] = -INFINITY;
    }
    constexpr int kUnroll = NPT == 2 ? MPCB_UNROLL_ROWS : MPCB_UNROLL4;
    for (int iv = 0; iv < nv; ++iv) {
        const float4 *__restrict__ row = tab + 2 * iv * ppr;
        const float rv = row[1].x;                         // r of the row
        float2 DV[NPT];
#pragma unroll
        for (int k = 0; k < NPT; ++k) { const float d = __fmaf_rn(-kWd2f, rv, nD[k]); DV[k] = make_float2(d, d); }
#pragma unroll kUnroll
        for (int i = 0; i < ppr; ++i) {
            const float4 t0 = row[2 * i];
            const float2 G = reinterpret_cast<const float2 *>(row + 2 * i + 1)[1];
            const float2 A = make_float2(t0.x, t0.y), B = make_float2(t0.z, t0.w);
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const float2 ndd = __ffma2_rn(U[k], A, __ffma2_rn(W[k], B, DV[k]));                    // -dd
                const float2 q = __ffma2_rn(NU[k], A, __ffma2_rn(NW[k], B, E[k]));
                float2 t = __ffma2_rn(make_float2(-q.x, -q.y), q, C[k]);
                if (HEAD) { const float2 gg = __fadd2_rn(G, Hh[k]); t = __ffma2_rn(make_float2(-gg.x, -gg.y), gg, t); }
                const float2 df = __ffma2_rn(t, t, ndd);
                m[k] = fmaxf(m[k], fmaxf(df.x, df.y));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) mx[k] = m[k];
}

// Stage 1 of the two-stage screen (option screen = 2, mpcb_screen.cuh): the same walk over the row table, forming only
// -dd -- the same operands and operations as prefix_screen_loop_rows, so the very same values -- and keeping its maximum
// per node: 2 FFMA2 + 1 FMNMX3 per node and leaf pair.  The line and heading terms enter through a per-node bound
// (screen_stage1_tmax).  Every lane reads the same pair at the same time, so the pairs' (a, b) come from the kernel
// parameter `ab` (RowPairs): the uniform datapath loads them (LDCU.64 into uniform registers, which the FFMA2s take as
// operands) instead of an LDS.128 writing the same four values into every lane's registers: 5 register writes per lane,
// node and pair instead of 7.  ptxas emits them only in code it knows the whole warp runs together (see the skip test
// of prefixn_kernel), and in small probes only while the loads are not addressed from the row counter, hence the two
// pointers that advance by themselves.  Each load feeds all NPT nodes of the lane: per 7 pairs, 14 LDCU.64 and the loop's
// bookkeeping serve 28 FFMA2 with two nodes per thread and 56 with four.  Only u2s, w2s and D2s of `p` are read.
template <int NPT>
__device__ __forceinline__ void prefix_dist_loop_rows(const RowPairs &ab, const float4 *__restrict__ tab, int nv, int ppr,
                                                      const ParentRegs (&p)[NPT], float (&mx)[NPT]) {
    float2 U[NPT], W[NPT];
    float nD[NPT], m[NPT];
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
        U[k] = make_float2(-p[k].u2s, -p[k].u2s); W[k] = make_float2(-p[k].w2s, -p[k].w2s);
        nD[k] = -p[k].D2s;
        m[k] = -INFINITY;
    }
    constexpr int kUnroll = MPCB_UNROLL_DIST;
    const float4 *__restrict__ row = tab;
    const float4 *pair = ab.ab;
    for (int iv = 0; iv < nv; ++iv, row += 2 * ppr, pair += ppr) {
        const float rv = row[1].x;
        float2 DV[NPT];
#pragma unroll
        for (int k = 0; k < NPT; ++k) { const float d = __fmaf_rn(-kWd2f, rv, nD[k]); DV[k] = make_float2(d, d); }
#pragma unroll kUnroll
        for (int i = 0; i < ppr; ++i) {
            const float4 t0 = pair[i];
            const float2 A = make_float2(t0.x, t0.y), B = make_float2(t0.z, t0.w);
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const float2 ndd = __ffma2_rn(U[k], A, __ffma2_rn(W[k], B, DV[k]));                    // -dd
                m[k] = fmaxf(m[k], fmaxf(ndd.x, ndd.y));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) mx[k] = m[k];
}

// scalar flavour on the same pair table: NEAR regime, or a node sitting exactly on the line origin
template <bool HEAD>
__device__ __forceinline__ float prefix_min_loop_scalar(const float4 *__restrict__ tab, int npairs, const ParentRegs &pr,
                                                        bool near, bool special, float Lspecial, float best) {
    for (int m = 0; m < npairs; ++m) {
        const float4 t0 = tab[2 * m], t1 = tab[2 * m + 1];
        float L0 = near ? leaf_val<HEAD, true>(t0.x, t0.z, t1.x, t1.z, pr) : leaf_val<HEAD, false>(t0.x, t0.z, t1.x, t1.z, pr);
        float L1 = near ? leaf_val<HEAD, true>(t0.y, t0.w, t1.y, t1.w, pr) : leaf_val<HEAD, false>(t0.y, t0.w, t1.y, t1.w, pr);
        if (special && t1.x == 0.f) L0 = Lspecial;
        if (special && t1.y == 0.f) L1 = Lspecial;
        best = fminf(best, fminf(L0, L1));
    }
    return best;
}

// PRUNE (pass 1 only): exact branch-and-bound.  While a node is set up, a lower bound on the cost of all its
// children is compared with the solve's running upper bound; nodes that provably cannot reach the refinement
// window are skipped lane by lane (a queue that compacts the survivors across tiles was measured 1.3-4x SLOWER:
// it serialises the float64 set-up and the fp32 pair loop that otherwise overlap between warps).
template <int PASS, bool HEAD, bool PRUNE = false, bool QMODE = false>
// (PASS is 1: the refinement pass of the prefix algorithm is refine_prefix_kernel)
__global__ void __launch_bounds__((PASS == 1 && !PRUNE) ? kPrefixCta : kThreads, (PASS == 1 && !PRUNE) ? 1 : 4)
prefix_kernel(const LaunchArgs a) {
    static_assert(PASS == 1, "pass 2 of the prefix algorithm is refine_prefix_kernel");
    extern __shared__ float4 s_leaf[];
    const int tid = threadIdx.x;
    const int S = a.g.S;
    const bool single = S <= kLeafChunk;
    // pass 1 stages the PAIR table (2 float4 per 2 leaves), pass 2 the plain per-leaf table;
    // either way a chunk of kLeafChunk leaves is kLeafChunk float4
    const float4 *__restrict__ gtab = PASS == 1 ? a.g.leaf32p : a.g.leaf32;
    auto chunk_f4 = [&](int cn) { return PASS == 1 ? 2 * ((cn + 1) >> 1) : cn; };
    if (single) {
        for (int i = tid; i < chunk_f4(S); i += blockDim.x) s_leaf[i] = __ldg(gtab + i);
        __syncthreads();
    }
    // pass 1: one work item = kPrefixCta/kThreads consecutive 256-node tiles of one solve, one per thread group;
    // pass 2: one work item = one listed tile (256 threads)
    // (the exhaustive kernel runs 1024-thread CTAs = 4 groups; the pruned one 256-thread CTAs = 1 group, so that a
    //  fully cut tile costs nothing more than its set-up)
    const unsigned groups = blockDim.x / kThreads;
    const unsigned long long qps = (a.tiles_per_solve + groups - 1) / groups;
    // QMODE (a separate instantiation, so that the tile walk keeps its registers): walk the children of the frontier's survivors
    constexpr bool qmode = PASS == 1 && PRUNE && QMODE;
    const bool listed = PASS == 1 && PRUNE && !QMODE && a.tile_list != nullptr;     // walk the survivors of tilecut_kernel
    if (PASS == 1 && PRUNE && gate_closed(a)) return;
    const unsigned qrounds = (unsigned)((S + kThreads - 1) / kThreads);   // 256-node rounds per depth-(H-2) node
    if (qmode && blockIdx.x == 0 && tid == 0) atomicAdd(a.counters + 2, a.counters[3]);   // subtrees the descent cut
    const unsigned long long nwork =
        qmode ? (unsigned long long)min(*a.q_count, a.q_cap) * qrounds
        : listed ? (unsigned long long)(*a.tile_count)
                 : PASS == 1 ? (unsigned long long)a.N * qps : (unsigned long long)(*a.work_count) * a.tps;
    // nodes this warp cut (statistics): kept in a register and added to the global counter ONCE, after the loop -- one
    // atomic per warp and tile on the same address (360k per cfg2 step) was what the pruned pass 1 waited for
    unsigned long long cut_acc = 0;
    for (unsigned long long w = blockIdx.x; w < nwork; w += gridDim.x) {
        unsigned seg; long long n; unsigned long long tile_lo, tile_hi;
        unsigned long long p_q = 0; bool in_q = false;                    // frontier mode: this thread's node
        if (qmode) {
            const unsigned long long e = w / qrounds;
            const unsigned c = (unsigned)(w - e * qrounds) * kThreads + tid;
            const unsigned long long g = a.q_list[e];
            n = (long long)a.fd[1].div(g);                                // fd[1].d = S^(H-2)
            p_q = (g - (unsigned long long)n * a.fd[1].d) * (unsigned long long)S + c;
            in_q = c < (unsigned)S;
            tile_lo = in_q ? (p_q - a.u_begin) / kThreads : 0;            // per lane
            tile_hi = tile_lo + 1;
            seg = (unsigned)((unsigned long long)n * a.segs_per_solve + (a.tps == 1 ? tile_lo : tile_lo / a.tps));
        } else if (listed) {
            const unsigned long long g = a.tile_list[w];
            n = (long long)a.fd_tiles.div(g);
            tile_lo = g - (unsigned long long)n * a.tiles_per_solve;
            tile_hi = tile_lo + 1;
            seg = (unsigned)((unsigned long long)n * a.segs_per_solve + (a.tps == 1 ? tile_lo : tile_lo / a.tps));
        } else if (PASS == 1) {
            n = (long long)(w / qps);
            const unsigned long long tile = (w - (unsigned long long)n * qps) * groups + (tid / kThreads);
            tile_lo = tile;
            tile_hi = tile < a.tiles_per_solve ? tile + 1 : tile;          // groups past the last tile idle
            seg = (unsigned)((unsigned long long)n * a.segs_per_solve + (a.tps == 1 ? tile : tile / a.tps));
        } else {
            decode_work<PASS>(a, w, seg, n, tile_lo, tile_hi);
        }
        const SolveParams &P = a.sp[n];
        if (P.flags & kFlagSkip) continue;               // a robot that has already stopped (uniform per work item)
        const bool origin_case = (P.flags & kFlagStartIsOrigin) != 0;
        double segbest = INFINITY;
        {
            const unsigned long long tile = tile_lo;
            const unsigned long long p = qmode ? p_q : a.u_begin + tile * kThreads + (tid % kThreads);
            const bool in_range = qmode ? in_q : (tile < tile_hi && p < a.u_end);
            ParentRegs pr = {};
            bool near = false, unmoved = false;
            double base = 0.0, base_direct = 0.0, lb = -INFINITY;
            bool active = in_range;
            // Pruned pass 1: an fp32 pre-filter first (float walk, the same bound in float, a margin of 8 tol1 -- it only
            // drops nodes the float64 test below would drop as well, mpcb_bounds.cuh), because all but a fraction of a per
            // cent of the nodes of a listed tile are nowhere near the bound and the float64 set-up is most of this kernel.
            unsigned pre_cut = 0;
            if (PASS == 1 && PRUNE && a.prefilter) {
                bool far = false;
                if (active) {
                    const double bound = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1 + P.tol;
                    far = node_far32(a, P, p, bound);
                }
                pre_cut = __ballot_sync(0xffffffffu, far);
                if (far) active = false;
            }
            // the node's frame and the bound over its children; the fp32 registers only for nodes that survive
            NodeFrame f;
            if (active) { node_frame(a, P, p, f); unmoved = f.unmoved; lb = node_lower_bound(a, P, f); }
            if (PASS == 1 && PRUNE) {
                const double bound = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1 + P.tol;
                const bool cut = active && lb > bound;
                const unsigned m = __ballot_sync(0xffffffffu, cut) | pre_cut;
                cut_acc += (unsigned)__popc(m);
                active = active && !cut;
            }
            // a warp none of whose nodes survived has nothing to score, publish or tighten (almost every warp of a listed
            // tile: the rest of the iteration is warp-level only when the table is resident, so the warp may leave it)
            if (PASS == 1 && PRUNE && single && !__any_sync(0xffffffffu, active)) continue;
            if (active) base = node_regs(a, f, pr, near, PASS == 1 ? &base_direct : nullptr);
            const bool special = active && origin_case && unmoved;
            if (PASS == 1 && !(near || special)) base = base_direct;   // the packed loop ranks in the direct form
            float best = INFINITY;
            const float Lspecial = (float)(P.special - 0.25 * (double)pr.e2 * (double)pr.e2);
            // chunked tables: a tile whose nodes were all cut must not stream the table through shared memory
            const bool any_active = (PASS == 1 && PRUNE && !single) ? (__syncthreads_or(active) != 0) : true;
            for (int c0 = 0; any_active && c0 < S; c0 += kLeafChunk) {
                const int cn = min(kLeafChunk, S - c0);
                if (!single) {
                    __syncthreads();
                    for (int i = tid; i < chunk_f4(cn); i += blockDim.x) s_leaf[i] = __ldg(gtab + c0 + i);
                    __syncthreads();
                }
                if (PASS == 1 && PRUNE) {
                    // After the cut the survivors are a few scattered lanes per warp (the promising nodes are a few steering
                    // directions per speed).  A lane running the pair loop on its own keeps the other 31 idle for S/2
                    // iterations, so sparse survivors are scored by the WHOLE warp instead, one node at a time with its
                    // leaf pairs spread over the lanes; dense warps keep one node per lane.
                    const int npairs = (cn + 1) >> 1;
                    const bool far_node = active && !(near || special);
                    unsigned coop = __ballot_sync(0xffffffffu, far_node);
                    if (__popc(coop) > 12) coop = 0;
                    const int lane = tid & 31;
                    for (unsigned todo = coop; todo; todo &= todo - 1) {
                        const int src = __ffs(todo) - 1;
                        float v = prefix_min_loop_far2_lanes<HEAD>(
                            s_leaf, npairs, __shfl_sync(0xffffffffu, pr.u2s, src), __shfl_sync(0xffffffffu, pr.w2s, src),
                            __shfl_sync(0xffffffffu, pr.D2s, src), __shfl_sync(0xffffffffu, pr.nu, src),
                            __shfl_sync(0xffffffffu, pr.nw, src), __shfl_sync(0xffffffffu, pr.eh, src),
                            __shfl_sync(0xffffffffu, pr.nhh, src), lane);
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
                        if (lane == src) best = fminf(best, v);
                    }
                    if (active && !((coop >> lane) & 1u))
                        best = (near || special) ? prefix_min_loop_scalar<HEAD>(s_leaf, npairs, pr, near, special, Lspecial, best)
                                                 : prefix_min_loop_far2<HEAD>(s_leaf, npairs, pr, best);
                    continue;
                }
                if (!active) continue;
                {
                    const int npairs = (cn + 1) >> 1;
                    best = (near || special) ? prefix_min_loop_scalar<HEAD>(s_leaf, npairs, pr, near, special, Lspecial, best)
                                             : prefix_min_loop_far2<HEAD>(s_leaf, npairs, pr, best);
                }
            }
            if (PASS == 1 && active) segbest = fmin(segbest, base + (double)best);
            if (PASS == 1 && PRUNE) {
                // tighten the solve's upper bound: this tile's best fp32 value + its error bound is >= a true leaf cost
                const double v = warp_min(active ? base + (double)best : INFINITY);
                if ((tid & 31) == 0 && v < INFINITY) atomicMin(a.ub + n, ordered_key(v + 0.5 * P.tol1));
            }
        }
        if (qmode) publish_segmin_lanes(a, seg, segbest);
        else publish_segmin(a, seg, segbest);
    }
    if (PASS == 1 && PRUNE && (tid & 31) == 0 && cut_acc) atomicAdd(a.counters + 2, cut_acc);
}

// ------------------------------------------------------------------------------------ prefix, pass 2 (refinement filter)
// The listed tiles, WARP BY WARP: a work item is one 32-node slice of a listed 256-node tile.  Of those 32 nodes only
// the few whose bound reaches into the window are live, and the warp scans them one at a time with the node's S leaves
// spread over its lanes (a lane scanning its node alone kept the other 31 idle for S iterations; the warp-wide scan never
// does more iterations than that).  In-window leaves go to the candidate list (or, if it is full, are evaluated on the
// spot and folded into the solve's record under its lock).  No CTA barrier: with a whole tile per CTA seven of eight
// warps waited at the barrier for the one that had something to scan (barrier stall 20 per issue, 9 % issue slots).
__device__ __forceinline__ void publish_best_warp(const LaunchArgs &a, long long n, double bJ, long long bj) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oJ = __shfl_xor_sync(0xffffffffu, bJ, o);
        const long long oj = __shfl_xor_sync(0xffffffffu, bj, o);
        lex_min(bJ, bj, oJ, oj);
    }
    // A result that is not lexicographically below the record cannot change it -- the record only ever decreases -- so it
    // does not queue for the lock (with one publish per listed node, or millions of exactly tied leaves, thousands of
    // warps took turns at the lock of the same solve).  The look without the lock is safe because of the order of the
    // accesses: the writer stores the index, fences, then stores the cost; the reader loads the cost, fences, then loads
    // the index.  The index it sees is therefore that of the record whose cost it saw or of a LATER (smaller) record, and
    // either way the pair (cost, index) it compares with is >= some record that really existed.
    bool go = false;
    if ((threadIdx.x & 31) == 0 && bj >= 0) {
        const double rJ = *(volatile double *)(a.bestJ + n);
        __threadfence();
        const long long rj = *(volatile long long *)(a.bestIdx + n);
        go = !(bJ > rJ || (bJ == rJ && rj >= 0 && bj >= rj));
    }
    if (go) {
        while (atomicCAS(a.lock + n, 0, 1) != 0) {}
        __threadfence();
        double cJ = *(volatile double *)(a.bestJ + n);
        long long cj = *(volatile long long *)(a.bestIdx + n);
        lex_min(cJ, cj, bJ, bj);
        *(volatile long long *)(a.bestIdx + n) = cj;
        __threadfence();
        *(volatile double *)(a.bestJ + n) = cJ;
        __threadfence();
        atomicExch(a.lock + n, 0);
    }
}

// the S leaves of one node spread over the lanes of a warp: in-window leaves become candidates.  Those that do not fit
// the candidate list are evaluated in float64 on the spot -- from the node's float64 pose, which the warp computes once
// per node (H-1 of the H steps of every such leaf are the node's: a batch with tens of millions of in-window leaves, the
// 16 x 16 grid at H = 4, spent three quarters of its refinement re-walking them)
template <bool HEAD>
__device__ __forceinline__ void scan_node(const LaunchArgs &a, const SolveParams &P, const float4 *__restrict__ tab, int S,
                                          int lane, const ParentRegs &q, bool qnear, bool qspecial, float qLsp, float qthr,
                                          double qbase, unsigned long long qp, long long n, double &bJ, long long &bj,
                                          unsigned long long &cand_acc) {
    bool have_pose = false;
    double nx = 0.0, ny = 0.0, nphi = 0.0;
    for (int c0 = 0; c0 < S; c0 += 32) {                       // uniform trip count: the warp votes inside
        const int c = c0 + lane;
        bool hit = false;
        double jrel = 0.0;
        if (c < S) {
            const float4 t = tab[c];
            float L = qnear ? leaf_val<HEAD, true>(t.x, t.y, t.z, t.w, q) : leaf_val<HEAD, false>(t.x, t.y, t.z, t.w, q);
            if (qspecial && t.z == 0.f) L = qLsp;
            hit = L <= qthr;
            jrel = qbase + (double)L;
        }
        const unsigned hm = __ballot_sync(0xffffffffu, hit);
        if (!hm) continue;
        cand_acc += hit ? 1u : 0u;
        const long long j = (long long)(qp * (unsigned long long)S + (unsigned)c);
        // list them: one reservation per warp, and none at all once the list is full (tens of millions of in-window
        // leaves each taking a turn at the same counter were a third of the refinement of such a batch)
        bool listed = false;
        if (a.cand) {
            unsigned slot0 = a.cand_cap;
            if (lane == 0 && *(volatile unsigned *)a.cand_count < a.cand_cap) slot0 = atomicAdd(a.cand_count, (unsigned)__popc(hm));
            slot0 = __shfl_sync(0xffffffffu, slot0, 0);
            const unsigned slot = slot0 + (unsigned)__popc(hm & ((1u << lane) - 1u));
            if (hit && slot0 < a.cand_cap && slot < a.cand_cap) {
                Candidate cd;
                cd.j = j; cd.jrel = jrel; cd.n = (int)n; cd.pad = 0;
                a.cand[slot] = cd;
                listed = true;
            }
        }
        const bool need = hit && !listed;
        if (!__any_sync(0xffffffffu, need)) continue;
        if (a.refine && a.mode != 1 && !have_pose) { exact_node_pose(a, P, qp, nx, ny, nphi); have_pose = true; }
        if (need) {
            const double J = !a.refine ? P.Kbase + jrel
                             : a.mode != 1 ? exact_child_cost(a, P, nx, ny, nphi, (unsigned)c) : exact_cost(a, P, j, nullptr, nullptr);
            lex_min(bJ, bj, J, j);
        }
    }
}

// the candidates a warp counted, added to the statistics once per warp
__device__ __forceinline__ void flush_cand_count(const LaunchArgs &a, unsigned long long cand_acc) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand_acc += __shfl_xor_sync(0xffffffffu, cand_acc, o);
    if ((threadIdx.x & 31) == 0 && cand_acc) atomicAdd(a.counters + 1, cand_acc);
}

template <bool HEAD>
__global__ void __launch_bounds__(kThreads, 4) refine_prefix_kernel(const LaunchArgs a) {
    extern __shared__ float4 s_leaf[];
    const int tid = threadIdx.x, lane = tid & 31;
    const int S = a.g.S;
    const bool single = S <= kLeafChunk;
    if (single) {
        for (int i = tid; i < S; i += blockDim.x) s_leaf[i] = __ldg(a.g.leaf32 + i);
        __syncthreads();
    }
    // a table that does not fit shared memory is read through L1/L2 (the lanes of a scan read consecutive entries)
    const float4 *__restrict__ tab = single ? s_leaf : a.g.leaf32;
    constexpr unsigned wpt = kThreads / 32;                                  // 32-node slices per tile
    const unsigned long long nww = (unsigned long long)(*a.work_count) * a.tps * wpt;
    unsigned long long seg_acc = 0;          // refined segments (statistics), added to the global counter once per warp
    unsigned long long cand_acc = 0;         // in-window leaves (statistics), likewise
    // Work items are handed out by a counter, not by position: what a slice costs ranges from nothing (no live node) to
    // thousands of float64 evaluations, and with a fixed assignment a batch rich in in-window leaves ran on 5 warps per SM
    // (warps active 8.5 %) while the others had long finished.
    for (;;) {
        unsigned long long ww = 0;
        if (lane == 0) ww = atomicAdd(a.refine_ctr, 1ULL);
        ww = __shfl_sync(0xffffffffu, ww, 0);
        if (ww >= nww) break;
        const unsigned long long wt = ww / wpt;
        const unsigned sub = (unsigned)(ww - wt * wpt);
        unsigned seg; long long n; unsigned long long tile_lo, tile_hi;
        decode_work<2>(a, wt, seg, n, tile_lo, tile_hi);
        if (sub == 0 && (a.tps == 1 || wt % a.tps == 0)) seg_acc += 1;
        const SolveParams &P = a.sp[n];
        if (P.flags & kFlagSkip) continue;
        const double tau = a.tau[n];
        const unsigned long long p = a.u_begin + tile_lo * kThreads + sub * 32u + lane;
        bool active = tile_lo < tile_hi && p < a.u_end;
        // (the same fp32 pre-filter as in the pruned pass 1, against this pass's bound: it drops only nodes the float64
        //  test below drops as well)
        if (active && a.prefilter && node_far32(a, P, p, tau + P.tol)) active = false;
        if (!__any_sync(0xffffffffu, active)) continue;
        NodeFrame f;
        if (active) {
            node_frame(a, P, p, f);
            if (node_lower_bound(a, P, f) > tau + P.tol) active = false;      // no child can lie inside the window
        }
        unsigned todo = __ballot_sync(0xffffffffu, active);
        if (!todo) continue;
        ParentRegs pr = {};
        bool near = false;
        double base = 0.0;
        if (active) base = node_regs(a, f, pr, near, nullptr);
        const bool special = active && (P.flags & kFlagStartIsOrigin) && f.unmoved;
        const float thr = __double2float_ru(tau - base);
        const float Lspecial = (float)(P.special - 0.25 * (double)pr.e2 * (double)pr.e2);
        // The live nodes of a tile sit next to each other (a few steering angles of one speed), i.e. in one or two of
        // its eight slices: scanned where they are found, those warps were the whole kernel (SM active cycles min / avg /
        // max 87k / 192k / 319k).  They are listed instead and refine_scan_kernel spreads them over all warps.
        // The list is kept short (option node_list, default 2^15): a solve batch with more live nodes than that has enough
        // of them everywhere to keep every warp busy, and once the list is full (one plain load) nothing is reserved.
        // Nor is anything listed once the candidate list has run full: a batch with that many in-window leaves evaluates
        // them where they are found, and its nodes are no longer scarce.
        int use_list = 0;
        if (a.node_list) {                       // lane 0 decides for the warp (the branch below contains shuffles)
            if (lane == 0)
                use_list = *(volatile unsigned *)a.node_count < a.node_cap &&
                           !(a.cand && *(volatile unsigned *)a.cand_count >= a.cand_cap);
            use_list = __shfl_sync(0xffffffffu, use_list, 0);
        }
        if (use_list) {
            const unsigned cnt = (unsigned)__popc(todo);
            unsigned slot0 = 0;
            if (lane == 0) slot0 = atomicAdd(a.node_count, cnt);
            slot0 = __shfl_sync(0xffffffffu, slot0, 0);
            const unsigned slot = slot0 + (unsigned)__popc(todo & ((1u << lane) - 1u));
            const bool fits = slot0 + cnt <= a.node_cap;                     // uniform
            if (active && slot < a.node_cap) {
                RefineNode e;
                e.u = pr.u; e.w = pr.w; e.u2 = pr.u2; e.w2 = pr.w2; e.D2 = pr.D2; e.Dp = pr.Dp; e.nu = pr.nu; e.nw = pr.nw;
                e.e2 = pr.e2; e.h2 = pr.h2; e.thr = thr; e.Lspecial = Lspecial; e.base = base; e.p = p;
                e.n = fits ? (int)n : -1;                                    // overflow: reserved slots stay empty
                e.flags = (near ? 1u : 0u) | (special ? 2u : 0u);
                a.node_list[slot] = e;
            }
            if (fits) continue;
        }
        double bJ = INFINITY; long long bj = -1;
        for (; todo; todo &= todo - 1) {
            const int src = __ffs(todo) - 1;
            ParentRegs q;
            q.u = __shfl_sync(0xffffffffu, pr.u, src); q.w = __shfl_sync(0xffffffffu, pr.w, src);
            q.u2 = __shfl_sync(0xffffffffu, pr.u2, src); q.w2 = __shfl_sync(0xffffffffu, pr.w2, src);
            q.D2 = __shfl_sync(0xffffffffu, pr.D2, src); q.Dp = __shfl_sync(0xffffffffu, pr.Dp, src);
            q.nu = __shfl_sync(0xffffffffu, pr.nu, src); q.nw = __shfl_sync(0xffffffffu, pr.nw, src);
            q.e2 = __shfl_sync(0xffffffffu, pr.e2, src); q.h2 = __shfl_sync(0xffffffffu, pr.h2, src);
            const bool qnear = __shfl_sync(0xffffffffu, (int)near, src) != 0;
            const bool qspecial = __shfl_sync(0xffffffffu, (int)special, src) != 0;
            const float qLsp = __shfl_sync(0xffffffffu, Lspecial, src), qthr = __shfl_sync(0xffffffffu, thr, src);
            const double qbase = __shfl_sync(0xffffffffu, base, src);
            const unsigned long long qp = __shfl_sync(0xffffffffu, p, src);
            scan_node<HEAD>(a, P, tab, S, lane, q, qnear, qspecial, qLsp, qthr, qbase, qp, n, bJ, bj, cand_acc);
        }
        if (__any_sync(0xffffffffu, bj >= 0)) publish_best_warp(a, n, bJ, bj);
    }
    if (lane == 0 && seg_acc) atomicAdd(a.counters, seg_acc);
    flush_cand_count(a, cand_acc);
}

// The listed nodes, one warp each (all scans cost the same: S leaves over 32 lanes).
template <bool HEAD>
__global__ void __launch_bounds__(kThreads, 4) refine_scan_kernel(const LaunchArgs a) {
    extern __shared__ float4 s_leaf[];
    const int tid = threadIdx.x, lane = tid & 31;
    const int S = a.g.S;
    const bool single = S <= kLeafChunk;
    const unsigned count = min(*a.node_count, a.node_cap);
    if (count == 0) return;
    if (single) {
        for (int i = tid; i < S; i += blockDim.x) s_leaf[i] = __ldg(a.g.leaf32 + i);
        __syncthreads();
    }
    const float4 *__restrict__ tab = single ? s_leaf : a.g.leaf32;
    // every warp takes a contiguous run of the list (the filter appends the live nodes of a slice together, so a run is
    // mostly one solve) and carries its best across the nodes of a solve: one publish per solve and warp, not per node
    constexpr unsigned wpc = kThreads / 32;
    const unsigned warps = gridDim.x * wpc, wid = blockIdx.x * wpc + (tid >> 5);
    const unsigned per = (count + warps - 1) / warps;
    const unsigned i0 = min(count, wid * per), i1 = min(count, i0 + per);
    unsigned long long cand_acc = 0;
    long long cur_n = -1;
    double bJ = INFINITY; long long bj = -1;
    for (unsigned i = i0; i < i1; ++i) {
        const RefineNode e = a.node_list[i];                                 // the same entry on every lane
        if (e.n < 0) continue;
        if (e.n != cur_n) {
            if (__any_sync(0xffffffffu, bj >= 0)) publish_best_warp(a, cur_n, bJ, bj);
            cur_n = e.n; bJ = INFINITY; bj = -1;
        }
        ParentRegs q = {};
        q.u = e.u; q.w = e.w; q.u2 = e.u2; q.w2 = e.w2; q.D2 = e.D2; q.Dp = e.Dp; q.nu = e.nu; q.nw = e.nw;
        q.e2 = e.e2; q.h2 = e.h2;
        scan_node<HEAD>(a, a.sp[e.n], tab, S, lane, q, (e.flags & 1u) != 0, (e.flags & 2u) != 0, e.Lspecial, e.thr, e.base,
                        e.p, e.n, bJ, bj, cand_acc);
    }
    if (__any_sync(0xffffffffu, bj >= 0)) publish_best_warp(a, cur_n, bJ, bj);
    flush_cand_count(a, cand_acc);
}

// ------------------------------------------------------------------------------------ prefix, several nodes per thread
// Pass 1, exhaustive only (option "nodes_per_thread" = 2 or 4): a CTA of 1024/NPT threads covers the same four 256-node
// tiles as prefix_kernel<1>, thread t holding nodes t, t + 1024/NPT, ... of the work item (NPT = 4: two such CTAs per
// SM).  Same arithmetic per node, so the segment minima (and everything downstream) are bit-identical to the
// one-node kernel.  SCREEN (option screen): 0 = MUFU.SQRT per leaf, 1 = the screen loop, 2 = the screen in two stages
// (below; it needs the row table, and launch_pass runs grids whose row table does not fit one chunk with 1).
//
// The two-stage work item runs in three phases.  A: each node is set up and keeps only what stage 1 reads -- u2s, w2s,
// D2s and its stage-1 bound T (screen_stage1_tmax) -- and a class: inactive, stage 1, or direct (NEAR, or unmoved on
// the line origin: the scalar loop).  B: if any lane of the warp holds a stage-1 node, prefix_dist_loop_rows runs for
// all NPT slots (the other classes' values are ignored).  C: each node that stage 1 passes (0.045 % of the cfg2
// nodes) and each direct node is set up again -- the same code on the same inputs, so the very same registers -- and
// scored alone: the screen loop, then the MUFU loop if it flags a leaf; direct nodes as in the one-stage kernel.
// Holding only stage 1's registers through the loop is what lets four nodes per thread share each table load.
__host__ __device__ constexpr int prefixn_cta(int npt) { return npt == 2 ? MPCB_PN_CTA2 : kPrefixCta / npt; }

static_assert(sizeof(LaunchArgs) + sizeof(RowPairs) <= 32764, "prefixn_kernel's parameters exceed the launch limit");

template <bool HEAD, int NPT, int SCREEN = 0>
__global__ void __launch_bounds__(prefixn_cta(NPT), NPT / 2)
prefixn_kernel(const LaunchArgs a, const __grid_constant__ RowPairs ab) {
    extern __shared__ float4 s_leaf[];
    constexpr int kCta = prefixn_cta(NPT);
    const int tid = threadIdx.x;
    const int S = a.g.S;
    // the screened kernel stages the pair table BY SPEED ROW when that fits one chunk (prefix_screen_loop_rows); every
    // other loop reads the very same array as a flat list of nv * ppr pairs
    const bool rows = SCREEN && a.g.ppr > 0;
    const bool single = rows || S <= kLeafChunk;
    const float4 *__restrict__ gtab = rows ? a.g.leaf32r : a.g.leaf32p;
    auto chunk_f4 = [&](int cn) { return 2 * ((cn + 1) >> 1); };
    if (single) {
        for (int i = tid; i < (rows ? 2 * a.g.nv * a.g.ppr : chunk_f4(S)); i += blockDim.x) s_leaf[i] = __ldg(gtab + i);
        __syncthreads();
    }
    constexpr unsigned groups = kCta * NPT / kThreads;           // 256-node tiles per work item
    static_assert(kCta * NPT % kThreads == 0, "a work item is a whole number of tiles");
    const unsigned long long qps = (a.tiles_per_solve + groups - 1) / groups;
    const unsigned long long nwork = (unsigned long long)a.N * qps;
    // SCREEN == 2: nodes that passed stage 1 (statistics), added to the global counter once per warp after the loop
    unsigned long long stage2_acc = 0;
    for (unsigned long long w = blockIdx.x; w < nwork; w += gridDim.x) {
        const long long n = (long long)(w / qps);
        const unsigned long long tile0 = (w - (unsigned long long)n * qps) * groups;
        const SolveParams &P = a.sp[n];
        // one solve per work item, so the test is uniform per CTA; REDUX puts it in a uniform register, and the branch
        // on it leaves the rest of the item in code ptxas knows to be warp-converged (a plain branch on P.flags does
        // not, and the stage-1 loop then reads its table with per-lane LDC.64)
        if (__reduce_or_sync(0xffffffffu, (unsigned)P.flags & kFlagSkip)) continue;
        const bool origin_case = (P.flags & kFlagStartIsOrigin) != 0;
        // slot k of the thread: its node p (false: past the solve's last node) and the segment it publishes to
        auto slot = [&](int k, unsigned long long &p, unsigned &sg) {
            const unsigned node = tid + k * kCta;
            const unsigned long long tile = tile0 + node / kThreads;
            p = a.u_begin + tile * kThreads + (node % kThreads);
            sg = (unsigned)((unsigned long long)n * a.segs_per_solve + (a.tps == 1 ? tile : tile / a.tps));
            return tile < a.tiles_per_solve && p < a.u_end;
        };
        // SCREEN: no leaf whose value exceeds the solve's upper bound (the exact probe, tightened by every node that
        // found something) by more than the ranking window tol1 can be the minimum or enter the refinement window
        double ubw = INFINITY;
        if (SCREEN) ubw = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1;
        const int npairs_rows = a.g.nv * a.g.ppr;
        double v[NPT];                  // each node's value base + best (INFINITY: nothing to publish)
        double vhit = INFINITY;         // the least value of the nodes the screen loop flagged
#pragma unroll
        for (int k = 0; k < NPT; ++k) v[k] = INFINITY;
        if constexpr (SCREEN == 2) {
            // A: set-up, keeping what stage 1 reads
            ParentRegs s1[NPT] = {};
            float tmax[NPT];
            unsigned staged = 0, direct = 0;     // bit k: slot k is a stage-1 / a direct node
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                unsigned long long p;
                unsigned sg;
                tmax[k] = 0.f;
                if (!slot(k, p, sg)) continue;
                ParentRegs q;
                bool nr, um;
                double bd;
                parent_setup(a, P, p, q, nr, um, nullptr, &bd);
                if (nr || (origin_case && um)) { direct |= 1u << k; continue; }
                staged |= 1u << k;
                s1[k].u2s = q.u2s; s1[k].w2s = q.w2s; s1[k].D2s = q.D2s;
                tmax[k] = screen_stage1_tmax(a.g.sbox, HEAD, __double2float_ru(ubw - bd), q.nu, q.nw, q.eh, q.nhh);
            }
            // B: stage 1, under a warp-uniform test (ptxas feeds the loop from uniform registers only in converged code)
            unsigned rare = direct;
            if (__reduce_or_sync(0xffffffffu, staged)) {
                float mdd[NPT];
                prefix_dist_loop_rows<NPT>(ab, s_leaf, a.g.nv, a.g.ppr, s1, mdd);
#pragma unroll
                for (int k = 0; k < NPT; ++k)
                    if (((staged >> k) & 1u) && screen_stage1_pass(tmax[k], mdd[k])) { rare |= 1u << k; ++stage2_acc; }
            }
            // C: the nodes stage 1 passed and the direct ones, set up again and scored one at a time
            for (unsigned m = rare; m; m &= m - 1) {
                const int k = __ffs(m) - 1;
                unsigned long long p;
                unsigned sg;
                slot(k, p, sg);
                ParentRegs pr;
                bool near, unmoved;
                double bd;
                double base = parent_setup(a, P, p, pr, near, unmoved, nullptr, &bd);
                float best = INFINITY;
                if ((direct >> k) & 1u) {
                    const float Ls = (float)(P.special - 0.25 * (double)pr.e2 * (double)pr.e2);
                    best = prefix_min_loop_scalar<HEAD>(s_leaf, npairs_rows, pr, near, origin_case && unmoved, Ls, best);
                } else {
                    base = bd;
                    const ParentRegs one[1] = {pr};
                    const float cn[1] = {__double2float_ru(ubw - bd)};
                    float mx[1];
                    prefix_screen_loop_rows<HEAD, 1>(s_leaf, a.g.nv, a.g.ppr, one, cn, mx);
                    if (mx[0] > 0.f) {              // some leaf of the node has t^2 - dd > 0: it may matter
                        best = prefix_min_loop_far2<HEAD>(s_leaf, npairs_rows, pr, best);
                        vhit = fmin(vhit, base + (double)best);
                    }
                }
#pragma unroll
                for (int j = 0; j < NPT; ++j)
                    if (j == k) v[j] = base + (double)best;
            }
        } else {
            ParentRegs pr[NPT] = {};
            bool near[NPT], special[NPT], active[NPT];
            double base[NPT];
            float best[NPT], Lspecial[NPT], cn[NPT];
            bool all = true;
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                unsigned long long p;
                unsigned sg;
                active[k] = slot(k, p, sg);
                bool unmoved = false;
                near[k] = false; base[k] = 0.0; best[k] = INFINITY;
                double base_direct = 0.0;
                if (active[k]) base[k] = parent_setup(a, P, p, pr[k], near[k], unmoved, nullptr, &base_direct);
                special[k] = active[k] && origin_case && unmoved;
                if (!(near[k] || special[k])) base[k] = base_direct;
                Lspecial[k] = (float)(P.special - 0.25 * (double)pr[k].e2 * (double)pr[k].e2);
                cn[k] = SCREEN ? __double2float_ru(ubw - base_direct) : 0.f;
                all = all && active[k] && !near[k] && !special[k];
            }
            bool hit[NPT];
#pragma unroll
            for (int k = 0; k < NPT; ++k) hit[k] = false;
            for (int c0 = 0; c0 < S; c0 += kLeafChunk) {
                const int cn_ = min(kLeafChunk, S - c0);
                if (!single) {
                    __syncthreads();
                    for (int i = tid; i < chunk_f4(cn_); i += blockDim.x) s_leaf[i] = __ldg(gtab + c0 + i);
                    __syncthreads();
                }
                const int npairs = rows ? npairs_rows : (cn_ + 1) >> 1;
                if (all && SCREEN) {
                    float mx[NPT];
                    if (rows) prefix_screen_loop_rows<HEAD, NPT>(s_leaf, a.g.nv, a.g.ppr, pr, cn, mx);
                    else prefix_screen_loop_far2xN<HEAD, NPT>(s_leaf, npairs, pr, cn, mx);
#pragma unroll
                    for (int k = 0; k < NPT; ++k)       // some leaf of the node has t^2 - dd > 0: it may matter
                        if (mx[k] > 0.f) { best[k] = prefix_min_loop_far2<HEAD>(s_leaf, npairs, pr[k], best[k]); hit[k] = true; }
                } else if (all) {
                    prefix_min_loop_far2xN<HEAD, NPT>(s_leaf, npairs, pr, best);
                } else {
#pragma unroll
                    for (int k = 0; k < NPT; ++k) {
                        if (!active[k]) continue;
                        best[k] = (near[k] || special[k])
                                      ? prefix_min_loop_scalar<HEAD>(s_leaf, npairs, pr[k], near[k], special[k], Lspecial[k], best[k])
                                      : prefix_min_loop_far2<HEAD>(s_leaf, npairs, pr[k], best[k]);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                if (active[k]) v[k] = base[k] + (double)best[k];
                if (hit[k]) vhit = fmin(vhit, v[k]);
            }
        }
        if (SCREEN) {
            // a node that found something tightens the solve's upper bound for the work items still to come:
            // its best fp32 value + the error bound of that value is >= the true cost of a leaf
            if (__any_sync(0xffffffffu, vhit < INFINITY)) {
                vhit = warp_min(vhit);
                if ((tid & 31) == 0) atomicMin(a.ub + n, ordered_key(vhit + 0.5 * P.tol1));
            }
        }
        // SCREEN: a node whose best value lies above the bound cannot hold the minimum or an in-window leaf, whichever loop
        // scored it (nodes in the NEAR regime or on the line origin are not screened leaf by leaf) -- it publishes nothing.
        // Otherwise a share of a split tree that holds no leaf near the bound would build its refinement window around
        // such nodes: on the config.py tree the 16^4 exactly tied unmoved nodes of the v = 0 share, 2.3e7 candidates.
#pragma unroll
        for (int k = 0; k < NPT; ++k) {
            unsigned long long p;
            unsigned sg;
            slot(k, p, sg);
            publish_segmin(a, sg, (!SCREEN || v[k] <= ubw) ? v[k] : INFINITY);
        }
    }
    if (SCREEN == 2) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) stage2_acc += __shfl_xor_sync(0xffffffffu, stage2_acc, o);
        if ((tid & 31) == 0 && stage2_acc) atomicAdd(a.counters + 7, stage2_acc);
    }
}

// ------------------------------------------------------------------------------------ frontier descent (pruned pass 1)
// Branch-and-bound from the top (H >= 3): the frontier of depth-k nodes that may still hold the argmin is expanded
// to depth k+1 -- one thread per (survivor, child): float64 walk of the child's k+1 controls, bound over all leaves
// H-k-1 steps below it against the solve's running upper bound -- until depth H-2; pass 1 then sets up and scores
// only the children of those survivors.  Cut subtrees are never enumerated at all, which is what makes 1e15-leaf
// trees a matter of milliseconds when the bound bites.  Node ids are global: n * S^k + index, so a child is simply
// id * S + c.  The lists have a fixed capacity; a frontier that outgrows it raises *overflow, the remaining levels and
// pass 1 return at once, and the host (which reads that one flag) redoes pass 1 through the tile bound.
__global__ void __launch_bounds__(kThreads) frontier_expand_kernel(const LaunchArgs a, int k,
                                                                   const unsigned long long *__restrict__ src,
                                                                   const unsigned *src_count,
                                                                   unsigned long long *__restrict__ dst,
                                                                   unsigned *dst_count, unsigned *overflow) {
    if (*(volatile unsigned *)overflow) return;
    const unsigned long long S = (unsigned long long)a.g.S;
    const unsigned long long nsrc = src ? (unsigned long long)min(*src_count, a.q_cap) : (unsigned long long)a.N;
    const unsigned long long c_lo = src ? 0ULL : (unsigned long long)a.i0_begin;
    const unsigned long long nchild = src ? S : (unsigned long long)(a.i0_end - a.i0_begin);
    const unsigned long long total = nsrc * nchild;
    const FastDiv64 fdn = a.fd[a.H - 2 - k];           // divisor S^(k+1): child id -> (solve, node index at depth k+1)
    const int steps = a.H - (k + 1);                   // control steps below a depth-(k+1) node
    const unsigned long long below = a.fd[k + 1].d;    // S^(H-2-k) depth-(H-1) nodes below it
    const unsigned lane = threadIdx.x & 31u;
    unsigned long long cut = 0;
    for (unsigned long long t0 = blockIdx.x * (unsigned long long)kThreads + (threadIdx.x & ~31u); t0 < total;
         t0 += (unsigned long long)gridDim.x * kThreads) {
        const unsigned long long t = t0 + lane;
        bool keep = false;
        unsigned long long child = 0;
        if (t < total) {
            const unsigned long long e = t / nchild;
            child = (src ? src[e] : e) * S + (t - e * nchild + c_lo);
            const unsigned long long n = fdn.div(child);
            const SolveParams &P = a.sp[n];
            if (!(P.flags & kFlagSkip)) {
                unsigned long long rem = child - n * fdn.d;
                double xi = 0.0, eta = 0.0, psi = 0.0, cp = 1.0, sp = 0.0;
                for (int m = 0; m <= k; ++m) {         // digit m has weight S^(k-m) = fd[H-1-k+m].d
                    const FastDiv64 &fd = a.fd[a.H - 1 - k + m];
                    const unsigned long long i = fd.div(rem);
                    rem -= i * fd.d;
                    walk_step(ldg_d4(a.g.tab64 + i), xi, eta, psi, cp, sp);
                }
                const double bound = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1 + P.tol;
                keep = !(subtree_lower_bound(a, P, xi, eta, psi, cp, sp, steps) > bound);      // NaN bounds never cut
                if (!keep) cut += below;
            }
        }
        const unsigned mk = __ballot_sync(0xffffffffu, keep);
        if (mk) {
            unsigned base = 0;
            if (lane == 0) base = atomicAdd(dst_count, (unsigned)__popc(mk));
            base = __shfl_sync(0xffffffffu, base, 0);
            const unsigned slot = base + __popc(mk & ((1u << lane) - 1u));
            if (keep) {
                if (slot < a.q_cap) dst[slot] = child;
                else *overflow = 1u;
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) cut += __shfl_xor_sync(0xffffffffu, cut, o);
    if (lane == 0 && cut) atomicAdd(a.counters + 3, cut);
}

// ------------------------------------------------------------------------------------ subtree cut (pruned pass 1)
// Branch-and-bound one level up (H >= 3): one thread per 256-node tile.  The tile's depth-(H-1) nodes are children of
// one depth-(H-2) node q (or of the few q the tile straddles); if the bound over ALL leaves two steps below every
// such q exceeds the solve's running upper bound, no node of the tile can hold a leaf inside the refinement window
// and the tile never reaches pass 1 (no set-up of its 256 nodes).  Survivors go to a list of global tile numbers that
// the pruned pass-1 kernels then walk.  Exactness: same argument as the per-node cut (DESIGN.md 3.4).
// does 256-node tile g (global tile number n * tiles_per_solve + tile) survive the depth-(H-2) bound?
__device__ __forceinline__ bool tile_survives(const LaunchArgs &a, unsigned long long g, unsigned &cut_nodes) {
    const unsigned long long n = a.fd_tiles.div(g), tile = g - n * a.tiles_per_solve;
    const SolveParams &P = a.sp[n];
    cut_nodes = 0;
    if (P.flags & kFlagSkip) return false;
    const unsigned long long p_lo = a.u_begin + tile * kThreads;
    const unsigned long long p_hi = min(p_lo + (unsigned long long)kThreads, a.u_end);     // exclusive
    const double bound = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1 + P.tol;
    bool keep = false;
    const unsigned long long q_hi = a.fd_S.div(p_hi - 1);
    for (unsigned long long q = a.fd_S.div(p_lo); q <= q_hi && !keep; ++q) {
        // the fp32 pre-filter first (mpcb_bounds.cuh, two steps): all but a few per cent of the tiles are nowhere near the
        // bound, and a tile it drops the float64 test below drops too
        if (a.prefilter) {
            const Prefilter32 pf = prefilter32(a, P);
            float xi = 0.f, eta = 0.f, psi = 0.f, cp = 1.f, sp = 0.f;
            parent_digits(a, q, [&](unsigned i) {
                const float4 t = __ldg(a.g.tab32 + i);
                walk_step_t<float>(t.x, t.y, t.z, t.w, xi, eta, psi, cp, sp);
            });
            if (node_prefilter32(pf, xi, eta, psi, cp, sp, 2) > __double2float_ru(bound + 8.0 * P.tol1)) continue;
        }
        double xi = 0.0, eta = 0.0, psi = 0.0, cp = 1.0, sp = 0.0;
        parent_digits(a, q, [&](unsigned i) { walk_step(ldg_d4(a.g.tab64 + i), xi, eta, psi, cp, sp); });
        keep = !(subtree_lower_bound(a, P, xi, eta, psi, cp, sp, 2) > bound);      // NaN bounds never cut
    }
    if (!keep) cut_nodes = (unsigned)(p_hi - p_lo);
    return keep;
}

__global__ void __launch_bounds__(kThreads) tilecut_kernel(const LaunchArgs a, unsigned long long g_begin,
                                                           unsigned long long g_end, unsigned long long *list,
                                                           unsigned *count, unsigned long long list_cap) {
    const unsigned long long g = g_begin + blockIdx.x * (unsigned long long)kThreads + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    bool keep = false;
    unsigned cut_nodes = 0;
    if (g < g_end) keep = tile_survives(a, g, cut_nodes);
    const unsigned mk = __ballot_sync(0xffffffffu, keep);
    unsigned base = 0;
    if (lane == 0 && mk) base = atomicAdd(count, (unsigned)__popc(mk));
    base = __shfl_sync(0xffffffffu, base, 0);
    // every launch tests at most list_cap tiles (one batch), so the list cannot overflow; the guard keeps a future
    // change of the batching from turning into an out-of-bounds store
    const unsigned long long slot = (unsigned long long)base + __popc(mk & ((1u << lane) - 1u));
    if (keep && slot < list_cap) list[slot] = g;
    for (int o = 16; o > 0; o >>= 1) cut_nodes += __shfl_xor_sync(0xffffffffu, cut_nodes, o);
    if (lane == 0 && cut_nodes) atomicAdd(a.counters + 2, (unsigned long long)cut_nodes);
}

// Fallback of the frontier descent, decided ON THE DEVICE: when a frontier outgrew its list (*q_overflow != 0), this
// kernel redoes pass 1 over all tiles -- tile bound and pruned pass 1 fused, no list in global memory, no host in the
// loop; when it did not, the kernel returns at once (the price of never synchronising: one empty launch).
// Work item = 256 consecutive tiles: every thread tests one tile (as tilecut_kernel does), the survivors are compacted
// into shared memory, then the CTA runs the pruned pass 1 on each of them (node-level cut lane by lane, pair loop,
// segment minimum, upper-bound tightening) -- the arithmetic of prefix_kernel<1, HEAD, true>.
template <bool HEAD>
__global__ void __launch_bounds__(kThreads, 4) tilewalk_fallback_kernel(const LaunchArgs a, unsigned long long all_tiles) {
    if (*(volatile const unsigned *)a.q_overflow == 0) return;
    extern __shared__ float4 s_leaf[];
    __shared__ unsigned long long s_tiles[kThreads];
    __shared__ unsigned s_warp[kThreads / 32];
    const int tid = threadIdx.x;
    const unsigned lane = tid & 31u, warp = tid >> 5;
    const int S = a.g.S;
    const bool single = S <= kLeafChunk;
    const float4 *__restrict__ gtab = a.g.leaf32p;
    auto chunk_f4 = [&](int cn) { return 2 * ((cn + 1) >> 1); };
    if (single) {
        for (int i = tid; i < chunk_f4(S); i += blockDim.x) s_leaf[i] = __ldg(gtab + i);
        __syncthreads();
    }
    if (blockIdx.x == 0 && tid == 0) a.counters[3] = 0;          // what the abandoned descent had counted as cut
    const unsigned long long items = (all_tiles + kThreads - 1) / kThreads;
    unsigned long long cut_acc = 0;          // nodes cut (statistics): lane 0's copy goes to the global counter after the loop
    for (unsigned long long w = blockIdx.x; w < items; w += gridDim.x) {
        const unsigned long long g = w * kThreads + tid;
        unsigned cut_nodes = 0;
        const bool keep = g < all_tiles && tile_survives(a, g, cut_nodes);
        const unsigned mk = __ballot_sync(0xffffffffu, keep);
        __syncthreads();                                          // the previous item's list has been consumed
        if (lane == 0) s_warp[warp] = __popc(mk);
        for (int o = 16; o > 0; o >>= 1) cut_nodes += __shfl_xor_sync(0xffffffffu, cut_nodes, o);
        cut_acc += cut_nodes;
        __syncthreads();
        unsigned before = 0, total = 0;
        for (unsigned i = 0; i < kThreads / 32; ++i) { if (i < warp) before += s_warp[i]; total += s_warp[i]; }
        if (keep) s_tiles[before + __popc(mk & ((1u << lane) - 1u))] = g;
        __syncthreads();
        for (unsigned t = 0; t < total; ++t) {
            const unsigned long long gt = s_tiles[t];
            const long long n = (long long)a.fd_tiles.div(gt);
            const unsigned long long tile = gt - (unsigned long long)n * a.tiles_per_solve;
            const unsigned seg = (unsigned)((unsigned long long)n * a.segs_per_solve + (a.tps == 1 ? tile : tile / a.tps));
            const SolveParams &P = a.sp[n];
            const unsigned long long p = a.u_begin + tile * kThreads + tid;
            bool active = p < a.u_end;
            ParentRegs pr = {};
            bool near = false, unmoved = false;
            double base = 0.0, base_direct = 0.0, lb = -INFINITY;
            if (active) base = parent_setup(a, P, p, pr, near, unmoved, &lb, &base_direct);
            const double bound = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1 + P.tol;
            const bool cut = active && lb > bound;
            const unsigned mc = __ballot_sync(0xffffffffu, cut);
            cut_acc += (unsigned)__popc(mc);
            active = active && !cut;
            const bool special = active && (P.flags & kFlagStartIsOrigin) && unmoved;
            if (!(near || special)) base = base_direct;
            const float Lspecial = (float)(P.special - 0.25 * (double)pr.e2 * (double)pr.e2);
            float best = INFINITY;
            const bool any_active = single ? true : (__syncthreads_or(active) != 0);
            for (int c0 = 0; any_active && c0 < S; c0 += kLeafChunk) {
                const int cn = min(kLeafChunk, S - c0);
                if (!single) {
                    __syncthreads();
                    for (int i = tid; i < chunk_f4(cn); i += blockDim.x) s_leaf[i] = __ldg(gtab + c0 + i);
                    __syncthreads();
                }
                if (!active) continue;
                const int npairs = (cn + 1) >> 1;
                best = (near || special) ? prefix_min_loop_scalar<HEAD>(s_leaf, npairs, pr, near, special, Lspecial, best)
                                         : prefix_min_loop_far2<HEAD>(s_leaf, npairs, pr, best);
            }
            const double v = active ? base + (double)best : INFINITY;
            const double vw = warp_min(v);
            if (lane == 0 && vw < INFINITY) atomicMin(a.ub + n, ordered_key(vw + 0.5 * P.tol1));
            publish_segmin(a, seg, v);
        }
    }
    if (lane == 0 && cut_acc) atomicAdd(a.counters + 2, cut_acc);
}

// ------------------------------------------------------------------------------------ prefix, pruned (pass 1)
// Exact branch-and-bound (option prune).  Cutting nodes lane by lane leaves warps with one or two live lanes --
// the promising nodes are scattered (a few steering directions per speed) -- so every WARP runs on its own:
// it sets up 32 nodes at a time in float64, tests each node's lower bound against the solve's running upper bound,
// appends the survivors to a warp-private shared-memory queue, and whenever 32 survivors are queued (and at the
// end) hands one to each lane and runs the dense pair loop.  The pair table is read straight from global memory
// (warp-uniform addresses, L1/L2 hits: ~6 % slower per pair than shared memory, tools/ubench/mix2.cu) so that no
// CTA barrier ties the warps together.  Results are identical to the exhaustive kernel.
struct __align__(8) QEntry {
    ParentRegs pr;
    float Lspecial;
    unsigned seg;
    double base;
    long long n;
    unsigned flags;      // bit0 near, bit1 special
    unsigned pad;
};
constexpr int kWarpQueue = 64;

template <bool HEAD, bool QMODE = false>
__global__ void __launch_bounds__(kThreads, 4) prefix_pruned_kernel(const LaunchArgs a) {
    extern __shared__ unsigned char s_raw[];
    QEntry *q = reinterpret_cast<QEntry *>(s_raw) + (threadIdx.x >> 5) * kWarpQueue;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const int S = a.g.S, npairs = (S + 1) >> 1;
    const float4 *__restrict__ tab = a.g.leaf32p;
    int count = 0;                                            // queue fill (warp-uniform)

    auto drain = [&](int m) {
        if (lane < m) {
            const QEntry e = q[lane];
            const float best = e.flags ? prefix_min_loop_scalar<HEAD>(tab, npairs, e.pr, (e.flags & 1) != 0,
                                                                      (e.flags & 2) != 0, e.Lspecial, INFINITY)
                                       : prefix_min_loop_far2<HEAD>(tab, npairs, e.pr, INFINITY);
            const double v = e.base + (double)best;
            if (v < INFINITY) {
                atomicMin(reinterpret_cast<unsigned long long *>(a.segmin) + e.seg, ordered_key(v));
                // this node's best fp32 value + its error bound is >= a true leaf cost: tighten the upper bound
                atomicMin(a.ub + e.n, ordered_key(v + 0.5 * a.sp[e.n].tol1));
            }
        }
        __syncwarp();
        const int rest = count - m;                           // < 32: move the tail to the front
        QEntry t;
        if (lane < rest) t = q[m + lane];
        __syncwarp();
        if (lane < rest) q[lane] = t;
        __syncwarp();
        count = rest;
    };

    const unsigned long long wtps = (a.u_end - a.u_begin + 31) / 32;      // 32-node warp tiles per solve
    constexpr bool qmode = QMODE;                                         // walk the children of the frontier's survivors
    const bool listed = !QMODE && a.tile_list != nullptr;                 // walk the survivors of tilecut_kernel
    if (gate_closed(a)) return;
    if (qmode && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(a.counters + 2, a.counters[3]);
    const unsigned qchunks = (unsigned)((S + 31) / 32);                   // 32-node chunks per depth-(H-2) node
    const unsigned long long nww = qmode ? (unsigned long long)min(*a.q_count, a.q_cap) * qchunks
                                   : listed ? (unsigned long long)(*a.tile_count) * (kThreads / 32)
                                            : (unsigned long long)a.N * wtps;
    const unsigned long long gw = (unsigned long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
    const unsigned long long GW = (unsigned long long)gridDim.x * (kThreads / 32);
    unsigned long long cut_acc = 0;          // nodes cut (statistics): one atomic per warp after the loop, not one per step
    for (unsigned long long ww = gw; ww < nww; ww += GW) {
        long long n; unsigned long long wt = 0, p_q = 0; bool in_q = false;
        if (qmode) {
            const unsigned long long e = ww / qchunks;
            const unsigned c = (unsigned)(ww - e * qchunks) * 32 + lane;
            const unsigned long long g = a.q_list[e];
            n = (long long)a.fd[1].div(g);
            p_q = (g - (unsigned long long)n * a.fd[1].d) * (unsigned long long)S + c;
            in_q = c < (unsigned)S;
        } else if (listed) {
            const unsigned long long g = a.tile_list[ww / (kThreads / 32)];
            n = (long long)a.fd_tiles.div(g);
            wt = (g - (unsigned long long)n * a.tiles_per_solve) * (kThreads / 32) + ww % (kThreads / 32);
            if (wt >= wtps) continue;                                     // ragged last tile
        } else {
            n = (long long)(ww / wtps);
            wt = ww - (unsigned long long)n * wtps;
        }
        const SolveParams &P = a.sp[n];
        if (P.flags & kFlagSkip) continue;
        const unsigned long long p = qmode ? p_q : a.u_begin + wt * 32 + lane;
        const bool in_range = qmode ? in_q : p < a.u_end;
        const unsigned long long tile = in_range ? (p - a.u_begin) / kThreads : 0;       // per lane
        const unsigned seg = (unsigned)((unsigned long long)n * a.segs_per_solve + (a.tps == 1 ? tile : tile / a.tps));
        ParentRegs pr = {};
        bool near = false, unmoved = false;
        double base = 0.0, base_direct = 0.0, lb = -INFINITY;
        if (in_range) base = parent_setup(a, P, p, pr, near, unmoved, &lb, &base_direct);
        const double bound = ordered_value(*(volatile unsigned long long *)(a.ub + n)) + P.tol1 + P.tol;
        const bool cut = in_range && lb > bound;
        const bool keep = in_range && !cut;
        const unsigned mk = __ballot_sync(0xffffffffu, keep), mc = __ballot_sync(0xffffffffu, cut);
        cut_acc += (unsigned)__popc(mc);
        if (keep) {
            QEntry e;
            e.pr = pr;
            e.Lspecial = (float)(P.special - 0.25 * (double)pr.e2 * (double)pr.e2);
            e.seg = seg; e.n = n;
            e.flags = (near ? 1u : 0u) | (((P.flags & kFlagStartIsOrigin) && unmoved) ? 2u : 0u);
            e.base = e.flags ? base : base_direct;
            e.pad = 0;
            q[count + __popc(mk & lt)] = e;
        }
        __syncwarp();
        count += __popc(mk);
        if (count >= 32) drain(32);
    }
    if (count > 0) drain(count);
    if (lane == 0 && cut_acc) atomicAdd(a.counters + 2, cut_acc);
}

// ------------------------------------------------------------------------------------ leafwalk
// One thread per leaf: decode the control sequence, walk H steps in registers in the start frame
// (heading relative to the start heading, so sin.approx/cos.approx see |psi| <~ 1), score.
// KIND: 0 = FULL with 64-bit leaf indices, 1 = FULL with every index < 2^32, 2 = HELD (control j held).
// SMEM: ctl points into shared memory (FULL trees whose {dphi, s} table fits).
// HT > 0: horizon known at compile time (the walk is fully unrolled, divisors live in uniform registers);
// HT = 0: run-time horizon a.H.
// fp32 leaf part of the leaf at (xi, eta, psi): the form pass 2 filters with, or (DIRECT) the one pass 1 ranks with.
// ORIGIN: 1 = the solve starts on the line origin (the reference's special case applies to leaves that have not
// moved), 0 = it does not, -1 = decide from P.flags per leaf.
template <bool HEAD, bool DIRECT, int ORIGIN = -1>
__device__ __forceinline__ float leafwalk_score(const SolveParams &P, const ParentRegs &pr, float xi, float eta,
                                                float psi, float Lsp) {
    const bool origin = ORIGIN < 0 ? (P.flags & kFlagStartIsOrigin) != 0 : ORIGIN != 0;
    const float g = 3.16227766016837952f * psi;
    if (DIRECT) {
        float L = leaf_walk_direct<HEAD>(xi, eta, psi, pr);
        if (origin && xi == 0.f && eta == 0.f)                               // the leaf has not moved off the line origin
            L = Lsp + (HEAD ? g * (g - pr.h2) : 0.f);
        return L;
    }
    const float r = __fmaf_rn(xi, xi, eta * eta);
    float L = (P.flags & kFlagNear) ? leaf_val<HEAD, true>(xi, eta, r, g, pr)
                                    : leaf_val<HEAD, false>(xi, eta, r, g, pr);
    if (origin && r == 0.f)
        L = Lsp + (HEAD ? g * (g - pr.h2) : 0.f);
    return L;
}

// DIRECT: rank with leaf_walk_direct (pass 1); Lsp is then the special-case value in the same units.
template <bool HEAD, int KIND, bool SMEM = false, int HT = 0, bool DIRECT = false>
__device__ __forceinline__ float leafwalk_eval(const LaunchArgs &a, const SolveParams &P, const ParentRegs &pr,
                                               const float2 *__restrict__ ctl, unsigned long long j,
                                               float &xi, float &eta, float &psi, float Lsp) {
    xi = 0.f; eta = 0.f; psi = 0.f;
    unsigned long long rem = j;
    unsigned rem32 = (unsigned)j;
    const int H = HT > 0 ? HT : a.H;
#pragma unroll
    for (int k = 0; k < (HT > 0 ? HT : kMaxH); ++k) {
        if (HT == 0 && k >= H) break;
        unsigned c;
        if (KIND == 2) c = (unsigned)j;
        else if (KIND == 1) { c = a.fd32[k].div(rem32); rem32 -= c * a.fd32[k].d; }
        else { unsigned long long q = a.fd[k].div(rem); rem -= q * a.fd[k].d; c = (unsigned)q; }
        float2 t = SMEM ? ctl[c] : __ldg(ctl + c);
        psi += t.x;
        float sn, cs;
        __sincosf(psi, &sn, &cs);
        xi = __fmaf_rn(t.y, cs, xi);
        eta = __fmaf_rn(t.y, sn, eta);
    }
    return leafwalk_score<HEAD, DIRECT>(P, pr, xi, eta, psi, Lsp);
}

// FULL tree, indices < 2^32, horizon HT known: the control digits of the thread's leaf are kept in registers and
// advanced by kThreads (mixed-radix add with carries) instead of being re-derived by divisions for every leaf.  The
// digits are kept PRE-SCALED as the addresses of their {dphi, s} table entries -- 32-bit shared-window addresses
// (SMEM: LDS.64 straight from the digit register; a generic pointer costs an LD.E and 64-bit address math) or byte
// offsets into the global table -- so that a step needs no address arithmetic at all.
template <bool HEAD, bool SMEM, int HT, bool ORIGIN>
__device__ __forceinline__ float leafwalk_eval_digits(const SolveParams &P, const ParentRegs &pr,
                                                      const float2 *__restrict__ ctl, const unsigned (&c)[HT], float Lsp) {
    float xi = 0.f, eta = 0.f, psi = 0.f;
#pragma unroll
    for (int k = 0; k < HT; ++k) {
        float2 t;
        if (SMEM)
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(t.x), "=f"(t.y) : "r"(c[k]));
        else
            t = __ldg(reinterpret_cast<const float2 *>(reinterpret_cast<const char *>(ctl) + c[k]));
        psi = k == 0 ? t.x : psi + t.x;
        float sn, cs;
        __sincosf(psi, &sn, &cs);
        xi = k == 0 ? t.y * cs : __fmaf_rn(t.y, cs, xi);
        eta = k == 0 ? t.y * sn : __fmaf_rn(t.y, sn, eta);
    }
    return leafwalk_score<HEAD, true, ORIGIN ? 1 : 0>(P, pr, xi, eta, psi, Lsp);      // pass 1 only: direct form
}

// the work loop of one CTA; HT as above
template <int PASS, bool HEAD, int KIND, int HT>
__device__ __forceinline__ void leafwalk_body(const LaunchArgs &a, const float2 *s_ctl, bool staged, double *s_J,
                                              long long *s_j) {
    const int tid = threadIdx.x;
    const unsigned long long nwork =
        PASS == 1 ? a.total_segs : (unsigned long long)(*a.work_count) * a.tps;
    for (unsigned long long w = blockIdx.x; w < nwork; w += gridDim.x) {
        unsigned seg; long long n; unsigned long long tile_lo, tile_hi;
        decode_work<PASS>(a, w, seg, n, tile_lo, tile_hi);
        const SolveParams &P = a.sp[n];
        if (P.flags & kFlagSkip) continue;
        ParentRegs pr;
        double base = start_as_parent(P, pr);
        double lsp = P.special - P.e0 * P.e0;                   // leaf part of an "on the line origin" leaf
        if (PASS == 1) {                                        // pass 1 ranks in the direct form: shift both
            const double off = start_direct_offset(P, pr);
            base = -off; lsp += off;
        }
        const float Lsp = (float)lsp;
        const bool smem = staged && !(P.flags & kFlagSlow);
        const float2 *ctl = smem ? s_ctl : ((P.flags & kFlagSlow) ? a.g.ctl32_slow : a.g.ctl32);
        const float thr = PASS == 2 ? __double2float_ru(a.tau[n] - base) : 0.f;
        if (PASS == 2 && tid == 0 && (a.tps == 1 || w % a.tps == 0)) atomicAdd(a.counters, 1ULL);
        float best = INFINITY;
        double bJ = INFINITY; long long bj = -1;
        for (unsigned long long tile = tile_lo; tile < tile_hi; ++tile) {
            const unsigned long long j0 = a.u_begin + tile * (unsigned long long)(kThreads * kLeafPerThread) + tid;
            if constexpr (PASS == 1 && KIND == 1 && HT > 0) {
                // digits of j0 once (as table addresses: base + 8 c), then +kThreads per leaf
                const unsigned S = (unsigned)a.g.S, jend = (unsigned)a.u_end;
                const unsigned base = smem ? (unsigned)__cvta_generic_to_shared(ctl) : 0u;
                const unsigned wrap = base + 8u * S;           // first address past the table
                unsigned c[HT], step[HT];
                unsigned rem32 = (unsigned)j0;
                bool step_low_only = true;                     // uniform: kThreads in base S has one digit
#pragma unroll
                for (int d = 0; d < HT; ++d) {
                    const unsigned q = a.fd32[d].div(rem32);
                    rem32 -= q * a.fd32[d].d;
                    c[d] = base + 8u * q;
                    step[d] = 8u * a.step_digits[d];
                    if (d < HT - 1) step_low_only = step_low_only && a.step_digits[d] == 0;
                }
                unsigned j32 = (unsigned)j0;
                // a tile that lies wholly inside the leaf range needs no per-leaf range test
                const bool whole = j0 + (unsigned long long)(kLeafPerThread - 1) * kThreads < a.u_end;
                // the table's address space, the line-origin special case, the shape of the index step and the range test
                // are uniform per launch, solve or tile: sixteen loops
                auto walk = [&](auto SM, auto ORG, auto LOW, auto WHOLE) {
#pragma unroll 4
                    for (int k = 0; k < kLeafPerThread; ++k) {
                        if (!decltype(WHOLE)::value && j32 >= jend) break;
                        best = fminf(best, leafwalk_eval_digits<HEAD, decltype(SM)::value, HT, decltype(ORG)::value>(
                                               P, pr, ctl, c, Lsp));
                        j32 += kThreads;
                        if (decltype(LOW)::value) {
                            // kThreads < S: only the last digit steps; the carry ripples further once in S leaves
                            unsigned v = c[HT - 1] + step[HT - 1];
                            if (v >= wrap) {
                                v -= 8u * S;
#pragma unroll
                                for (int d = HT - 2; d >= 0; --d) {
                                    c[d] += 8u;
                                    if (c[d] < wrap) break;
                                    c[d] = base;
                                }
                            }
                            c[HT - 1] = v;
                        } else {
                            unsigned carry = 0;
#pragma unroll
                            for (int d = HT - 1; d >= 0; --d) {
                                unsigned v = c[d] + step[d] + carry;
                                carry = v >= wrap ? 8u : 0u;
                                c[d] = v - (carry ? 8u * S : 0u);
                            }
                        }
                    }
                };
                using T = std::true_type; using F = std::false_type;
                const bool org = (P.flags & kFlagStartIsOrigin) != 0;
                auto pick2 = [&](auto SM, auto ORG, auto LOW) { if (whole) walk(SM, ORG, LOW, T{}); else walk(SM, ORG, LOW, F{}); };
                auto pick = [&](auto SM, auto ORG) { if (step_low_only) pick2(SM, ORG, T{}); else pick2(SM, ORG, F{}); };
                if (smem) { if (org) pick(T{}, T{}); else pick(T{}, F{}); }
                else      { if (org) pick(F{}, T{}); else pick(F{}, F{}); }
            } else {
                // kLeafPerThread leaves per thread, strided by the CTA width (coalesced table reads)
#pragma unroll 4
                for (int k = 0; k < kLeafPerThread; ++k) {
                    const unsigned long long j = j0 + (unsigned)k * kThreads;
                    if (j >= a.u_end) break;
                    float xi, eta, psi;
                    const float L = smem ? leafwalk_eval<HEAD, KIND, true, HT, PASS == 1>(a, P, pr, ctl, j, xi, eta, psi, Lsp)
                                         : leafwalk_eval<HEAD, KIND, false, HT, PASS == 1>(a, P, pr, ctl, j, xi, eta, psi, Lsp);
                    if (PASS == 1) best = fminf(best, L);
                    else if (L <= thr) take_candidate(a, P, n, (long long)j, base + (double)L, bJ, bj);
                }
            }
        }
        if (PASS == 1) publish_segmin(a, seg, base + (double)best);
        else publish_best(a, n, bJ, bj, s_J, s_j);
    }
}

template <int PASS, bool HEAD, int KIND>
__global__ void __launch_bounds__(kThreads) leafwalk_kernel(const LaunchArgs a) {
    extern __shared__ float2 s_ctl[];        // FULL trees: the {dphi, s} table, when it fits (a.lw_smem)
    __shared__ double s_J[kThreads / 32];
    __shared__ long long s_j[kThreads / 32];
    const bool staged = KIND != 2 && a.lw_smem;
    if (staged) {
        for (int i = threadIdx.x; i < a.g.S; i += kThreads) s_ctl[i] = __ldg(a.g.ctl32 + i);
        __syncthreads();
    }
    // pass 1 is specialised for the common horizons (the reference's 3, and 2/4); pass 2 is rare
    if (PASS == 1 && a.H == 3) leafwalk_body<PASS, HEAD, KIND, 3>(a, s_ctl, staged, s_J, s_j);
    else if (PASS == 1 && a.H == 4) leafwalk_body<PASS, HEAD, KIND, 4>(a, s_ctl, staged, s_J, s_j);
    else if (PASS == 1 && a.H == 2) leafwalk_body<PASS, HEAD, KIND, 2>(a, s_ctl, staged, s_J, s_j);
    else leafwalk_body<PASS, HEAD, KIND, 0>(a, s_ctl, staged, s_J, s_j);
}

// ------------------------------------------------------------------------------------ dump
// All leaves of solve 0 in [dump_begin, dump_begin+dump_count): {x, y, phi, L} as one 16-byte
// store per thread (consecutive threads -> consecutive leaves: fully coalesced STG.128).
template <bool HEAD>
__global__ void __launch_bounds__(kThreads) leafwalk_dump_kernel(const LaunchArgs a, double *jrel) {
    const SolveParams &P = a.sp[0];
    ParentRegs pr;
    const double base = start_as_parent(P, pr);
    const float2 *ctl = (P.flags & kFlagSlow) ? a.g.ctl32_slow : a.g.ctl32;
    const float c0 = (float)cos(P.phi0), s0 = (float)sin(P.phi0);
    const double off = a.dump_direct ? start_direct_offset(P, pr) : 0.0;      // what pass 1 ranks with, in its own units
    const float Lsp = (float)(P.special - P.e0 * P.e0 + off);
    for (unsigned long long i = blockIdx.x * (unsigned long long)kThreads + threadIdx.x; i < a.dump_count;
         i += (unsigned long long)gridDim.x * kThreads) {
        float xi, eta, psi;
        const unsigned long long j = a.dump_begin + i;
        const float L = a.dump_direct
                            ? (a.mode == 1 ? leafwalk_eval<HEAD, 2, false, 0, true>(a, P, pr, ctl, j, xi, eta, psi, Lsp)
                                           : leafwalk_eval<HEAD, 0, false, 0, true>(a, P, pr, ctl, j, xi, eta, psi, Lsp))
                            : (a.mode == 1 ? leafwalk_eval<HEAD, 2>(a, P, pr, ctl, j, xi, eta, psi, Lsp)
                                           : leafwalk_eval<HEAD, 0>(a, P, pr, ctl, j, xi, eta, psi, Lsp));
        a.dump[i] = make_float4((float)P.xs + (c0 * xi - s0 * eta), (float)P.ys + (s0 * xi + c0 * eta),
                                (float)P.phi0 + psi, L);
        jrel[i] = (a.dump_direct ? -off : base) + (double)L;
    }
}

// prefix flavour of the dump (test-only: strided stores): J_rel = base_p + L for every child
template <bool HEAD>
__global__ void __launch_bounds__(kThreads) prefix_dump_kernel(const LaunchArgs a, double *jrel) {
    const SolveParams &P = a.sp[0];
    const int S = a.g.S;
    const unsigned long long p_lo = a.dump_begin / S, p_hi = (a.dump_begin + a.dump_count + S - 1) / S;
    for (unsigned long long p = p_lo + blockIdx.x * (unsigned long long)kThreads + threadIdx.x; p < p_hi;
         p += (unsigned long long)gridDim.x * kThreads) {
        ParentRegs pr;
        bool near, unmoved;
        double base_direct;
        double base = parent_setup(a, P, p, pr, near, unmoved, nullptr, &base_direct);
        const bool special = (P.flags & kFlagStartIsOrigin) && unmoved;
        const float Lspecial = (float)(P.special - 0.25 * (double)pr.e2 * (double)pr.e2);
        const bool direct = a.dump_direct && !near && !special;      // what pass 1 ranks this node's children with
        if (direct) base = base_direct;
        for (int c = 0; c < S; ++c) {
            const unsigned long long j = p * S + c;
            if (j < a.dump_begin || j >= a.dump_begin + a.dump_count) continue;
            float4 t = __ldg(a.g.leaf32 + c);
            float L = direct ? leaf_val_direct<HEAD>(t.x, t.y, t.z, t.w, pr)
                      : near ? leaf_val<HEAD, true>(t.x, t.y, t.z, t.w, pr)
                             : leaf_val<HEAD, false>(t.x, t.y, t.z, t.w, pr);
            if (special && t.z == 0.f) L = Lspecial;
            jrel[j - a.dump_begin] = base + (double)L;
        }
    }
}

// ------------------------------------------------------------------------------------ small kernels
// Raw inputs -> SolveParams (float64), incl. the per-solve error window of the refinement pass.
__global__ void prep_kernel(long long N, const double *__restrict__ state, const double *__restrict__ target,
                            const double *__restrict__ origin, const double *__restrict__ threshold,
                            const uint8_t *__restrict__ flags, int cost_kind, int H, int kind,
                            double smax, double dphimax, double tol_scale, SolveParams *__restrict__ out) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= N) return;
    SolveParams P;
    P.xs = state[3 * n]; P.ys = state[3 * n + 1]; P.phi0 = state[3 * n + 2];
    P.xt = target[2 * n]; P.yt = target[2 * n + 1];
    P.ox = origin[2 * n]; P.oy = origin[2 * n + 1];
    P.theta = atan(P.xt / P.yt);
    P.lineA = P.yt - P.oy; P.lineB = P.xt - P.ox;
    P.lineC = __dadd_rn(__dmul_rn(P.xt, P.oy), -__dmul_rn(P.yt, P.ox));
    // rounded as the reference rounds it (no FMA contraction)
    P.line_norm = sqrt(__dadd_rn(__dmul_rn(P.lineA, P.lineA), __dmul_rn(P.lineB, P.lineB)));
    P.threshold = threshold ? threshold[n] : INFINITY;
    P.wl = cost_kind == 0 ? 10.0 : 100.0;
    P.wh = cost_kind == 0 ? 3.16227766016837952 : 0.0;
    P.inv_wl = 1.0 / P.wl;
    double s0, c0;
    sincos(P.phi0, &s0, &c0);
    const double rx = P.xt - P.xs, ry = P.yt - P.ys;
    P.u0 = c0 * rx + s0 * ry; P.w0 = c0 * ry - s0 * rx;
    P.d0 = sqrt(rx * rx + ry * ry);
    // the anchor of the fp32 line offsets: its rounding is part of the error model's world-coordinate term below
    const double E0 = __dadd_rn(__dadd_rn(__dmul_rn(P.lineA, P.xs), -__dmul_rn(P.lineB, P.ys)), P.lineC);
    P.e0 = P.wl * E0 / P.line_norm;
    P.nx0 = P.wl * (P.lineA * c0 - P.lineB * s0) / P.line_norm;
    P.ny0 = P.wl * (-P.lineA * s0 - P.lineB * c0) / P.line_norm;
    P.hp0 = P.wh * (P.theta - P.phi0);
    P.Kbase = kWd * P.d0 + P.e0 * P.e0 + P.hp0 * P.hp0;
    P.special = 1.0e6 * P.wl * P.wl;
    // kind: bit0 = prefix algorithm, bit1 = HELD tree.  The slow-down override belongs to the online (HELD)
    // controller (math_model_tree.py:312-316); FULL solves ignore the flag.
    const bool prefix = (kind & 1) != 0, held = (kind & 2) != 0;
    int f = (flags && held) ? (flags[n] & kFlagSlow) : 0;
    if (flags && (flags[n] & 2)) f |= kFlagSkip;          // MPCB_FLAG_SKIP
    if (P.xs == P.ox && P.ys == P.oy) f |= kFlagStartIsOrigin;
    // error model of the fp32 leaf part (DESIGN.md section 3.3)
    const double Rtot = H * smax;
    const double Rl = prefix ? smax : Rtot;
    const double Gl = P.wh * (prefix ? dphimax : H * dphimax);
    const bool near = !(P.d0 >= 4.0 * Rl);
    if (!prefix && near) f |= kFlagNear;
    const double E = fabs(P.e0) + P.wl * Rtot, Hh = fabs(P.hp0) + P.wh * H * dphimax, Q = P.wl * Rl;
    double M = kWd * Rl * 16.0 + 4.0 * Q * (2.0 * E + Q) + 4.0 * Gl * (Gl + 2.0 * Hh);
    // sin.approx / cos.approx: absolute error 2^-21.4 on [-pi, pi], growing with the argument beyond it
    if (!prefix) M += kWd * Rtot * 8.0 * fmax(1.0, H * dphimax / 3.141592653589793);
    // float64 rounding at the solve's coordinates (DESIGN.md section 3.3): the costs the window is compared with are the
    // reference's float64 ones, whose roundings grow with |x|, |y|, |phi|, while the fp32 offsets carry none of them
    //   heading after H steps: H roundings at |phi| <= Phi                                 -> dphi
    //   position after H steps: H roundings at |x| <= X, |y| <= Y, and s dphi per step     -> dp (both axes)
    //   line distance: 4 roundings of the sum at the size of its terms, and dp             -> de (scaled by wl)
    // each enters the reference's cost once and the anchors e0, hp0 of the fp32 form once
    const double Phi = fabs(P.phi0) + H * dphimax, X = fabs(P.xs) + Rtot, Y = fabs(P.ys) + Rtot;
    const double dphi = H * 1.1102230246251565e-16 * Phi;                       // 2^-53
    const double dp = H * 2.220446049250313e-16 * (X + Y) + H * smax * dphi;    // 2^-52
    const double lsum = fabs(P.lineA) * X + fabs(P.lineB) * Y + fabs(P.xt * P.oy) + fabs(P.yt * P.ox);
    const double de = P.wl * (4.440892098500626e-16 * lsum / P.line_norm + dp);  // 2^-51
    const double dh = P.wh * dphi;
    const double Mw = (kWd * dp + 2.0 * de * (2.0 * E + de) + 2.0 * dh * (2.0 * Hh + dh)) * 8388608.0;   // in 2^-23
    M += Mw;
    P.tol = 2.0 * M * 1.1920928955078125e-07 * tol_scale;
    P.tol1 = P.tol;
    if (prefix) {
        // direct form of the prefix pass 1 (leaf_val_direct), in units of 2^-23:
        //   distance   kWd d (sqrt.approx 1 + roundings of D2s, the FFMA chain under the root ~0.75) -> 3 kWd Dmax
        //   roundings of the table entries and of u2s, w2s                                            -> 2 kWd smax
        //   (q + eh)^2 with |q + eh| <= E1: 1.5 ulp on the sum, squared                                -> 4 E1^2
        //   (g + nhh)^2 with |g + nhh| <= H1                                                           -> 3 H1^2
        //   the two accumulating FFMAs round at the magnitude of the whole value (half an ulp each)    -> Vmax
        const double Dmax = P.d0 + Rtot, E1 = E + Q, H1 = Hh + Gl;
        const double Vmax = kWd * Dmax + E1 * E1 + H1 * H1;
        const double M1 = 3.0 * kWd * Dmax + 2.0 * kWd * smax + 4.0 * E1 * E1 + 3.0 * H1 * H1 + Vmax + Mw;
        P.tol1 = fmax(P.tol, 2.0 * M1 * 1.1920928955078125e-07 * tol_scale);
    } else {
        // direct form of the leafwalk pass 1 (leaf_walk_direct): the walk's own error (M) plus
        //   kWd d from dx, dy, their sum of squares and sqrt.approx, the rounding of kWd (u, w)   -> 4 kWd Dmax
        //   (q + eh)^2, (g + nhh)^2 and the two accumulating FFMAs as above                      -> 4 E1^2 + 3 H1^2 + Vmax
        const double Dmax = P.d0 + Rtot, E1 = E + Q, H1 = Hh + Gl;
        const double Vmax = kWd * Dmax + E1 * E1 + H1 * H1;
        const double M1 = M + 4.0 * kWd * Dmax + 4.0 * E1 * E1 + 3.0 * H1 * H1 + Vmax;
        P.tol1 = 2.0 * M1 * 1.1920928955078125e-07 * tol_scale;
    }
    P.flags = f; P.pad = 0;
    prefilter_solve_consts(P);
    out[n] = P;
}

// Pruning probe (FULL): the S "held" sequences (c, c, ..., c) are leaves of the FULL tree, so the best of them,
// evaluated exactly, is an upper bound on the minimal cost: it seeds the branch-and-bound before pass 1.
__global__ void __launch_bounds__(kThreads) probe_kernel(const LaunchArgs a) {
    __shared__ double s_J[kThreads / 32];
    for (long long n = blockIdx.x; n < a.N; n += gridDim.x) {
        const SolveParams &P = a.sp[n];
        if (P.flags & kFlagSkip) { if (threadIdx.x == 0) a.ub[n] = ~0ULL; continue; }
        double best = INFINITY;
        // only sequences whose first control lies in this launch's share of the tree are leaves of it
        for (int c = a.i0_begin + threadIdx.x; c < a.i0_end; c += kThreads) {
            double x = P.xs, y = P.ys, phi = P.phi0;
            for (int k = 0; k < a.H; ++k) exact_step(a, a.g.tab64, a.g.vtab, c, x, y, phi);
            best = fmin(best, exact_terminal(a, P, x, y, phi));
        }
        best = warp_min(best);
        if ((threadIdx.x & 31) == 0) s_J[threadIdx.x >> 5] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int i = 1; i < kThreads / 32; ++i) best = fmin(best, s_J[i]);
            a.ub[n] = best < INFINITY ? ordered_key(best - P.Kbase) : ~0ULL;
        }
        __syncthreads();
    }
}

// Per solve: minimum of its segment minima -> window edge tau; segments inside the window -> work list.
__global__ void __launch_bounds__(kThreads) reduce_compact_kernel(const LaunchArgs a, double *tau,
                                                                  unsigned *worklist, unsigned *work_count) {
    __shared__ double s_J[kThreads / 32];
    __shared__ double s_tau;
    const unsigned sps = (unsigned)a.segs_per_solve;
    for (long long n = blockIdx.x; n < a.N; n += gridDim.x) {
        const unsigned long long *sm = reinterpret_cast<const unsigned long long *>(a.segmin) + (unsigned long long)n * sps;
        double v = INFINITY;
        for (unsigned i = threadIdx.x; i < sps; i += kThreads) v = fmin(v, ordered_value(sm[i]));
        v = warp_min(v);
        if ((threadIdx.x & 31) == 0) s_J[threadIdx.x >> 5] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int i = 1; i < kThreads / 32; ++i) v = fmin(v, s_J[i]);
            // the segment holding the true argmin has a pass-1 minimum <= v + tol1; its pass-2 value is <= v + (tol1+tol)/2
            s_tau = v + a.sp[n].tol1;
            tau[n] = v + 0.5 * (a.sp[n].tol1 + a.sp[n].tol);
            a.bestJ[n] = INFINITY;
            a.bestIdx[n] = -1;
            a.lock[n] = 0;
        }
        __syncthreads();
        const double t = s_tau;
        if (t < INFINITY)
            for (unsigned i = threadIdx.x; i < sps; i += kThreads)
                if (ordered_value(sm[i]) <= t) worklist[atomicAdd(work_count, 1u)] = (unsigned)(n * sps + i);
        __syncthreads();
    }
}

// The same in three grid-wide steps, for launches whose solves have many segments each (one oversized tree: 4e6
// segments scanned by ONE CTA took 5.8 of the 6.0 ms of a 1e15-leaf pruned solve):
//   (1) every CTA folds the minimum of a chunk of segment keys into its solve's key,
//   (2) one thread per solve turns that into the window edge and resets the solve's record,
//   (3) every CTA lists the qualifying segments of a chunk (warp-aggregated append; the order of the work list is
//       irrelevant -- pass 2 reduces lexicographically).
constexpr unsigned kReduceChunk = 4096;      // segment keys per CTA step

__global__ void __launch_bounds__(kThreads) segmin_fold_kernel(const LaunchArgs a, unsigned long long *solve_key) {
    const unsigned sps = (unsigned)a.segs_per_solve;
    const unsigned cps = (sps + kReduceChunk - 1) / kReduceChunk;          // chunks per solve
    const unsigned long long *keys = reinterpret_cast<const unsigned long long *>(a.segmin);
    for (unsigned long long w = blockIdx.x; w < (unsigned long long)a.N * cps; w += gridDim.x) {
        const unsigned long long n = w / cps;
        const unsigned lo = (unsigned)(w - n * cps) * kReduceChunk, hi = min(lo + kReduceChunk, sps);
        unsigned long long k = ~0ULL;
        for (unsigned i = lo + threadIdx.x; i < hi; i += kThreads) k = min(k, keys[n * sps + i]);
        for (int o = 16; o > 0; o >>= 1) k = min(k, __shfl_xor_sync(0xffffffffu, k, o));
        if ((threadIdx.x & 31) == 0 && k != ~0ULL) atomicMin(solve_key + n, k);
    }
}

__global__ void window_edge_kernel(const LaunchArgs a, const unsigned long long *solve_key, double *tau, double *tau1) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    const double v = ordered_value(solve_key[n]);                           // untouched key (all ones) -> NaN/inf: no segment
    const bool any = solve_key[n] != ~0ULL;
    tau1[n] = any ? v + a.sp[n].tol1 : -INFINITY;
    tau[n] = any ? v + 0.5 * (a.sp[n].tol1 + a.sp[n].tol) : -INFINITY;
    a.bestJ[n] = INFINITY;
    a.bestIdx[n] = -1;
    a.lock[n] = 0;
}

__global__ void __launch_bounds__(kThreads) seg_compact_kernel(const LaunchArgs a, const double *tau1, unsigned *worklist,
                                                               unsigned *work_count) {
    const unsigned sps = (unsigned)a.segs_per_solve;
    const unsigned cps = (sps + kReduceChunk - 1) / kReduceChunk;
    const unsigned long long *keys = reinterpret_cast<const unsigned long long *>(a.segmin);
    const unsigned lane = threadIdx.x & 31u;
    for (unsigned long long w = blockIdx.x; w < (unsigned long long)a.N * cps; w += gridDim.x) {
        const unsigned long long n = w / cps;
        const unsigned lo = (unsigned)(w - n * cps) * kReduceChunk, hi = min(lo + kReduceChunk, sps);
        const double t = tau1[n];
        for (unsigned i0 = lo + (threadIdx.x & ~31u); i0 < hi; i0 += kThreads) {
            const unsigned i = i0 + lane;
            const bool take = i < hi && ordered_value(keys[n * sps + i]) <= t;
            const unsigned mk = __ballot_sync(0xffffffffu, take);
            if (!mk) continue;
            unsigned base = 0;
            if (lane == 0) base = atomicAdd(work_count, (unsigned)__popc(mk));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (take) worklist[base + __popc(mk & ((1u << lane) - 1u))] = (unsigned)(n * sps + i);
        }
    }
}

// Refinement, second half: every listed candidate is evaluated in float64 by its own thread (reference formula and
// operation order, exact_cost), the smallest cost per solve is folded with an atomicMin on its order-preserving key ...
__global__ void __launch_bounds__(kThreads) cand_eval_kernel(const LaunchArgs a) {
    const unsigned count = min(*a.cand_count, a.cand_cap);
    for (unsigned i = blockIdx.x * kThreads + threadIdx.x; i < count; i += gridDim.x * kThreads) {
        const Candidate c = a.cand[i];
        const double J = a.refine ? exact_cost(a, a.sp[c.n], c.j, nullptr, nullptr) : (a.sp[c.n].Kbase + c.jrel);
        a.cand_J[i] = J;
        if (J == J) atomicMin(a.cand_key + c.n, ordered_key(J));         // NaN costs never win
    }
}

// ... then the lowest leaf index among the candidates of that cost (first minimum, math_model.py:195) ...
__global__ void __launch_bounds__(kThreads) cand_select_kernel(const LaunchArgs a) {
    const unsigned count = min(*a.cand_count, a.cand_cap);
    for (unsigned i = blockIdx.x * kThreads + threadIdx.x; i < count; i += gridDim.x * kThreads) {
        const Candidate c = a.cand[i];
        const double J = a.cand_J[i];
        if (J == J && ordered_key(J) == a.cand_key[c.n]) atomicMin(a.cand_idx + c.n, (unsigned long long)c.j);
    }
}

// ... and merged with what pass 2 evaluated on the spot (only when the list overflowed): the solve's record.
__global__ void cand_merge_kernel(const LaunchArgs a) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    double J = a.bestJ[n]; long long j = a.bestIdx[n];
    if (a.cand_key[n] != ~0ULL) lex_min(J, j, ordered_value(a.cand_key[n]), (long long)a.cand_idx[n]);
    a.bestJ[n] = J; a.bestIdx[n] = j;
}

// Winner -> outputs: float64 re-roll of its trajectory, threshold test (math_model.py:195).
__global__ void finalize_kernel(const LaunchArgs a, double *best_cost, long long *best_index, double *best_traj,
                                double *first_control) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    const SolveParams &P = a.sp[n];
    const long long j = a.bestIdx[n];
    double J = a.bestJ[n];
    double tr[3 * kMaxH];
    int c0 = 0;
    bool ok = j >= 0;
    if (ok) {
        const double Je = exact_cost(a, P, j, tr, &c0);
        if (a.refine) J = Je;
    } else {
        J = NAN;
    }
    if (best_cost) best_cost[n] = J;
    if (best_index) best_index[n] = (ok && J < P.threshold) ? j : -1;
    if (best_traj)
        for (int k = 0; k < 3 * a.H; ++k) best_traj[(size_t)n * 3 * a.H + k] = ok ? tr[k] : NAN;
    if (first_control) {
        const bool slow = (P.flags & kFlagSlow) != 0;
        first_control[2 * n] = ok ? (slow ? a.g.vtab_slow : a.g.vtab)[c0] : NAN;
        first_control[2 * n + 1] = ok ? a.g.beta[c0 % a.g.nb] : NAN;
    }
}

// Split tree (one tree shared by the ranks of a communicator): this rank's best leaf per solve -> 16-byte record ...
__global__ void split_pack_kernel(const LaunchArgs a, SplitRec *mine) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    mine[n].cost = a.bestJ[n];
    mine[n].index = a.bestIdx[n];
}

// ... and, after the all-gather, the lexicographic (cost, index) minimum over the ranks' records becomes the solve's
// record on EVERY rank (rank r's record of solve n is all[r * N + n]); finalize_kernel then re-rolls the winner's
// trajectory locally -- no broadcast.  NaN costs never win (math_model.py:195: a NaN cost fails the strict '<').
__global__ void split_pick_kernel(const LaunchArgs a, const SplitRec *all, int nranks) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    double bJ = INFINITY; long long bj = -1;
    for (int r = 0; r < nranks; ++r) {
        const SplitRec rec = all[(size_t)r * a.N + n];
        if (rec.cost == rec.cost) lex_min(bJ, bj, rec.cost, rec.index);
    }
    a.bestJ[n] = bJ;
    a.bestIdx[n] = bj;
}

// Split tree, before the descent: every rank's probe bounds the minimum of the WHOLE tree from above (its held
// sequences are leaves of it), so the ranks share their bounds -- all[r * N + n] = rank r's key of solve n -- and each
// continues with the smallest.  Without it a rank whose share holds no good leaf prunes against a weak bound.
__global__ void split_ub_min_kernel(const LaunchArgs a, const unsigned long long *all, int nranks) {
    const long long n = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    unsigned long long k = a.ub[n];
    for (int r = 0; r < nranks; ++r) k = min(k, all[(size_t)r * a.N + n]);
    a.ub[n] = k;
}

// ------------------------------------------------------------------------------------ launchers
cudaError_t launch_split_ub_min(cudaStream_t st, const LaunchArgs &a, const unsigned long long *all, int nranks) {
    split_ub_min_kernel<<<(unsigned)((a.N + 127) / 128), 128, 0, st>>>(a, all, nranks);
    return cudaGetLastError();
}

cudaError_t launch_split_pack(cudaStream_t st, const LaunchArgs &a, SplitRec *mine) {
    split_pack_kernel<<<(unsigned)((a.N + 127) / 128), 128, 0, st>>>(a, mine);
    return cudaGetLastError();
}

cudaError_t launch_split_pick(cudaStream_t st, const LaunchArgs &a, const SplitRec *all, int nranks) {
    split_pick_kernel<<<(unsigned)((a.N + 127) / 128), 128, 0, st>>>(a, all, nranks);
    return cudaGetLastError();
}

static inline int grid_for(unsigned long long work, int sms, int per_sm) {
    unsigned long long cap = (unsigned long long)sms * per_sm;
    return (int)(work < cap ? (work ? work : 1) : cap);
}

cudaError_t launch_prep(cudaStream_t st, long long N, const double *state, const double *target,
                        const double *origin, const double *threshold, const uint8_t *flags, int cost_kind, int H,
                        int prefix, double smax, double dphimax, double tol_scale, SolveParams *out) {
    const int bs = 128;
    prep_kernel<<<(unsigned)((N + bs - 1) / bs), bs, 0, st>>>(N, state, target, origin, threshold, flags, cost_kind,
                                                            H, prefix, smax, dphimax, tol_scale, out);
    return cudaGetLastError();
}

static size_t prefix_smem(const LaunchArgs &a) {
    const size_t rows = 2 * (size_t)a.g.nv * a.g.ppr;            // the row table (0 if it does not fit one chunk)
    const size_t flat = (size_t)(a.g.S < kLeafChunk ? a.g.S + 1 : kLeafChunk);
    return sizeof(float4) * (rows > flat ? rows : flat);
}

template <typename K>
static int resident_ctas(K kernel, size_t smem, int threads) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1) n = 1;
    return n;
}

template <typename K>
static cudaError_t launch_persistent(K kernel, const LaunchArgs &a, int pass, size_t smem, int sms, cudaStream_t st,
                                     int threads = kThreads, const RowPairs *ab = nullptr) {
    // pass 1: one CTA per resident slot, striding over the segments; pass 2: same grid over the
    // device-side work list (its length is not known on the host)
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int slots = sms * resident_ctas(kernel, smem, threads);
    const int grid = pass == 1 ? (int)(a.total_segs < (unsigned long long)slots ? a.total_segs : slots) : slots;
    if constexpr (std::is_invocable_v<K, const LaunchArgs, const RowPairs>) kernel<<<grid, threads, smem, st>>>(a, *ab);
    else kernel<<<grid, threads, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pass(cudaStream_t st, const LaunchArgs &a, const RowPairs &ab, int pass, bool prefix, int sms) {
    const bool head = a.cost_kind == 0;
    if (prefix) {
        const size_t sm = prefix_smem(a);
        if (pass == 1 && a.prune && a.g.S > kLeafChunk) {
            // big grids (table streamed in chunks): warp-private survivor queues -- config 0: 2.6 s -> 0.25 s per tick
            const size_t smq = sizeof(QEntry) * kWarpQueue * (kThreads / 32);
            if (a.q_list)
                return head ? launch_persistent(prefix_pruned_kernel<true, true>, a, pass, smq, sms, st)
                            : launch_persistent(prefix_pruned_kernel<false, true>, a, pass, smq, sms, st);
            return head ? launch_persistent(prefix_pruned_kernel<true>, a, pass, smq, sms, st)
                        : launch_persistent(prefix_pruned_kernel<false>, a, pass, smq, sms, st);
        }
        if (pass == 1 && a.prune && a.q_list)
            return head ? launch_persistent(prefix_kernel<1, true, true, true>, a, pass, sm, sms, st)
                        : launch_persistent(prefix_kernel<1, false, true, true>, a, pass, sm, sms, st);
        if (pass == 1 && a.prune)   // small grids: nodes are cut lane by lane (the queue costs more than it saves there)
            return head ? launch_persistent(prefix_kernel<1, true, true>, a, pass, sm, sms, st)
                        : launch_persistent(prefix_kernel<1, false, true>, a, pass, sm, sms, st);
#define MPCB_PN(NPT_, SCR_)                                                                                      \
    (head ? launch_persistent(prefixn_kernel<true, NPT_, SCR_>, a, pass, sm, sms, st, prefixn_cta(NPT_), &ab)    \
          : launch_persistent(prefixn_kernel<false, NPT_, SCR_>, a, pass, sm, sms, st, prefixn_cta(NPT_), &ab))
        // the two-stage screen needs the row table; without it the one-stage flat loop runs
        const int scr = a.screen == 2 && a.g.ppr == 0 ? 1 : a.screen;
        if (pass == 1 && a.npt == 4) return scr == 2 ? MPCB_PN(4, 2) : scr ? MPCB_PN(4, 1) : MPCB_PN(4, 0);
        if (pass == 1 && a.npt == 2) return scr == 2 ? MPCB_PN(2, 2) : scr ? MPCB_PN(2, 1) : MPCB_PN(2, 0);
#undef MPCB_PN
        if (pass == 1)
            return head ? launch_persistent(prefix_kernel<1, true>, a, pass, sm, sms, st, kPrefixCta)
                        : launch_persistent(prefix_kernel<1, false>, a, pass, sm, sms, st, kPrefixCta);
        const size_t sm2 = sizeof(float4) * (size_t)(a.g.S <= kLeafChunk ? a.g.S : 0);       // pass 2 stages the per-leaf table
        return head ? launch_persistent(refine_prefix_kernel<true>, a, pass, sm2, sms, st)
                    : launch_persistent(refine_prefix_kernel<false>, a, pass, sm2, sms, st);
    }
    const int kind = a.mode == 1 ? 2 : (a.idx32 ? 1 : 0);
    const size_t lw_sm = (a.mode != 1 && a.lw_smem) ? sizeof(float2) * (size_t)a.g.S : 0;
#define MPCB_LW(P_, H_, K_) launch_persistent(leafwalk_kernel<P_, H_, K_>, a, pass, lw_sm, sms, st)
#define MPCB_LW_KIND(P_, H_) (kind == 2 ? MPCB_LW(P_, H_, 2) : kind == 1 ? MPCB_LW(P_, H_, 1) : MPCB_LW(P_, H_, 0))
    if (pass == 1) return head ? MPCB_LW_KIND(1, true) : MPCB_LW_KIND(1, false);
    return head ? MPCB_LW_KIND(2, true) : MPCB_LW_KIND(2, false);
#undef MPCB_LW_KIND
#undef MPCB_LW
}

cudaError_t launch_frontier_expand(cudaStream_t st, const LaunchArgs &a, int k, const unsigned long long *src,
                                   const unsigned *src_count, unsigned long long *dst, unsigned *dst_count,
                                   unsigned *overflow, int sms) {
    frontier_expand_kernel<<<sms * 8, kThreads, 0, st>>>(a, k, src, src_count, dst, dst_count, overflow);
    return cudaGetLastError();
}

cudaError_t launch_tilecut(cudaStream_t st, const LaunchArgs &a, unsigned long long g_begin, unsigned long long g_end,
                           unsigned long long *list, unsigned *count, unsigned long long list_cap) {
    if (g_end - g_begin > list_cap) return cudaErrorInvalidValue;
    const unsigned long long blocks = (g_end - g_begin + kThreads - 1) / kThreads;
    tilecut_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(a, g_begin, g_end, list, count, list_cap);
    return cudaGetLastError();
}

cudaError_t launch_tilewalk_fallback(cudaStream_t st, const LaunchArgs &a, unsigned long long all_tiles, int sms) {
    const size_t sm = prefix_smem(a);
    const bool head = a.cost_kind == 0;
    auto go = [&](auto kernel) {
        const int grid = sms * resident_ctas(kernel, sm, kThreads);
        kernel<<<grid, kThreads, sm, st>>>(a, all_tiles);
        return cudaGetLastError();
    };
    return head ? go(tilewalk_fallback_kernel<true>) : go(tilewalk_fallback_kernel<false>);
}

cudaError_t launch_probe(cudaStream_t st, const LaunchArgs &a, int sms) {
    probe_kernel<<<grid_for((unsigned long long)a.N, sms, 8), kThreads, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_reduce_compact(cudaStream_t st, const LaunchArgs &a, double *tau, unsigned *worklist,
                                  unsigned *work_count, int sms) {
    reduce_compact_kernel<<<grid_for((unsigned long long)a.N, sms, 8), kThreads, 0, st>>>(a, tau, worklist,
                                                                                         work_count);
    return cudaGetLastError();
}

// the grid-wide flavour; scratch = 2 * N 8-byte words (solve keys, pass-1 window edges)
cudaError_t launch_reduce_compact_wide(cudaStream_t st, const LaunchArgs &a, double *tau, unsigned *worklist,
                                       unsigned *work_count, void *scratch, int sms, int *launches) {
    unsigned long long *solve_key = static_cast<unsigned long long *>(scratch);
    double *tau1 = reinterpret_cast<double *>(solve_key + a.N);
    cudaError_t e = cudaMemsetAsync(solve_key, 0xFF, sizeof(unsigned long long) * a.N, st);
    if (e != cudaSuccess) return e;
    const unsigned long long chunks = (unsigned long long)a.N * ((a.segs_per_solve + kReduceChunk - 1) / kReduceChunk);
    const int grid = grid_for(chunks, sms, 8);
    segmin_fold_kernel<<<grid, kThreads, 0, st>>>(a, solve_key);
    window_edge_kernel<<<(unsigned)((a.N + 127) / 128), 128, 0, st>>>(a, solve_key, tau, tau1);
    seg_compact_kernel<<<grid, kThreads, 0, st>>>(a, tau1, worklist, work_count);
    *launches += 3;
    return cudaGetLastError();
}

cudaError_t launch_refine_scan(cudaStream_t st, const LaunchArgs &a, int sms) {
    const size_t sm2 = sizeof(float4) * (size_t)(a.g.S <= kLeafChunk ? a.g.S : 0);
    return a.cost_kind == 0 ? launch_persistent(refine_scan_kernel<true>, a, 2, sm2, sms, st)
                            : launch_persistent(refine_scan_kernel<false>, a, 2, sm2, sms, st);
}

cudaError_t launch_cand_resolve(cudaStream_t st, const LaunchArgs &a, int sms) {
    cand_eval_kernel<<<sms * 4, kThreads, 0, st>>>(a);
    cand_select_kernel<<<sms * 4, kThreads, 0, st>>>(a);
    cand_merge_kernel<<<(unsigned)((a.N + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_finalize(cudaStream_t st, const LaunchArgs &a, double *best_cost, long long *best_index,
                            double *best_traj, double *first_control) {
    const int bs = 128;
    finalize_kernel<<<(unsigned)((a.N + bs - 1) / bs), bs, 0, st>>>(a, best_cost, best_index, best_traj,
                                                                  first_control);
    return cudaGetLastError();
}

cudaError_t launch_dump(cudaStream_t st, const LaunchArgs &a, bool prefix, double *jrel, int sms) {
    const bool head = a.cost_kind == 0;
    if (prefix) {
        const unsigned long long parents = a.dump_count / a.g.S + 2;
        const int grid = grid_for((parents + kThreads - 1) / kThreads, sms, 8);
        if (head) prefix_dump_kernel<true><<<grid, kThreads, 0, st>>>(a, jrel);
        else prefix_dump_kernel<false><<<grid, kThreads, 0, st>>>(a, jrel);
    } else {
        const int grid = grid_for((a.dump_count + kThreads - 1) / kThreads, sms, 8);
        if (head) leafwalk_dump_kernel<true><<<grid, kThreads, 0, st>>>(a, jrel);
        else leafwalk_dump_kernel<false><<<grid, kThreads, 0, st>>>(a, jrel);
    }
    return cudaGetLastError();
}

}  // namespace mpcb
