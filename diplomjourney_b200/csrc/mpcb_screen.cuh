// mpcb_screen.cuh -- stage 1 of the two-stage screen of the exhaustive prefix pass 1 (option screen = 2, DESIGN.md 3.5).
//
// The screen (prefix_screen_loop_rows, stage 2) flags a node iff one of its leaves has fma(t, t, -dd) > 0, where
//      dd = the leaf's scaled squared distance,   q = fma(nu, a, fma(nw, b, eh)),   gg = g + nhh   (HEAD only),
//      t  = fma(-gg, gg, fma(-q, q, cn)),
// all in fp32, round to nearest.  Stage 1 forms only dd for every leaf (prefix_dist_loop_rows) and bounds t per node:
// every step above is a correctly rounded operation, and a correctly rounded operation is monotone in each operand, so
//  * over the box [amin, amax] x [bmin, bmax] x [gmin, gmax] of the table's fp32 (a, b, g), the fp32 q of every leaf
//    lies in [qlo, qhi] -- the same two FMAs on the box corners that minimise / maximise them -- and gg in
//    [fl(gmin + nhh), fl(gmax + nhh)];
//  * fl(c - x^2) does not increase with |x|, so the same two FMAs on the value of each interval nearest to 0 give an
//    upper bound thi, and on the value farthest from 0 a lower bound tlo, on the t of every leaf of the node;
//  * t^2 <= T^2 with T = max(|thi|, |tlo|), and fma(t, t, -dd) = fl(t^2 - dd) does not decrease with t^2 or with -dd.
// Hence fma(T, T, max(-dd)) >= fma(t, t, -dd) for every leaf: a node whose stage-1 value is <= 0 holds no leaf stage 2
// would flag -- neither a real hit (t > 0) nor a false one (t < 0, t^2 > dd), so the nodes re-run in full, the values
// published and the upper bound's tightening are those of the one-stage screen.  No slack is needed: the bound replays
// the kernel's own roundings instead of bounding them.  A NaN anywhere makes the stage-1 value NaN, and a NaN passes.
//
// Host/device, so that tests/test_screen_stage1_on_host.py compiles exactly this code with g++.
#pragma once
#include <cmath>

#if defined(__CUDACC__)
#define MPCB_SCR_HD __host__ __device__ __forceinline__
#else
#define MPCB_SCR_HD inline
#endif

namespace mpcb {

// The range of the fp32 control table's a = s cos dphi, b = s sin dphi and g = sqrt(10) dphi over all S controls
// (GridTables::leaf32, which every pair table repeats): a grid constant, set with the tables.
struct ScreenBox {
    float amin, amax, bmin, bmax, gmin, gmax;
};

MPCB_SCR_HD float scr_fma(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
    return __fmaf_rn(a, b, c);
#else
    return std::fma(a, b, c);
#endif
}

MPCB_SCR_HD float scr_add(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}

// the value of [lo, hi] nearest to 0, and one farthest from 0
MPCB_SCR_HD float scr_near0(float lo, float hi) { return lo > 0.f ? lo : (hi < 0.f ? hi : 0.f); }
MPCB_SCR_HD float scr_far0(float lo, float hi) { return std::fabs(lo) > std::fabs(hi) ? lo : hi; }

// [lo, hi] holding the fp32 q = fma(nu, a, fma(nw, b, eh)) of every (a, b) of the box, and the fp32 gg = g + nhh
MPCB_SCR_HD void screen_q_range(const ScreenBox &bx, float nu, float nw, float eh, float &lo, float &hi) {
    const float ilo = scr_fma(nw, nw >= 0.f ? bx.bmin : bx.bmax, eh), ihi = scr_fma(nw, nw >= 0.f ? bx.bmax : bx.bmin, eh);
    lo = scr_fma(nu, nu >= 0.f ? bx.amin : bx.amax, ilo);
    hi = scr_fma(nu, nu >= 0.f ? bx.amax : bx.amin, ihi);
}
MPCB_SCR_HD void screen_g_range(const ScreenBox &bx, float nhh, float &lo, float &hi) {
    lo = scr_add(bx.gmin, nhh);
    hi = scr_add(bx.gmax, nhh);
}

// [tlo, thi] holding the t = fma(-gg, gg, fma(-q, q, cn)) of every leaf of the node (cn, nu, nw, eh, nhh: the node's fp32
// screen bound and direct-form registers, exactly as the stage-2 loop reads them)
MPCB_SCR_HD void screen_t_range(const ScreenBox &bx, bool head, float cn, float nu, float nw, float eh, float nhh,
                                float &tlo, float &thi) {
    float qlo, qhi;
    screen_q_range(bx, nu, nw, eh, qlo, qhi);
    const float qn = scr_near0(qlo, qhi), qf = scr_far0(qlo, qhi);
    thi = scr_fma(-qn, qn, cn);
    tlo = scr_fma(-qf, qf, cn);
    if (head) {
        float glo, ghi;
        screen_g_range(bx, nhh, glo, ghi);
        const float gn = scr_near0(glo, ghi), gf = scr_far0(glo, ghi);
        thi = scr_fma(-gn, gn, thi);
        tlo = scr_fma(-gf, gf, tlo);
    }
}

// T = max(|thi|, |tlo|): |t| <= T for every leaf of the node.  NaN stays NaN.
MPCB_SCR_HD float screen_stage1_tmax(const ScreenBox &bx, bool head, float cn, float nu, float nw, float eh, float nhh) {
    float tlo, thi;
    screen_t_range(bx, head, cn, nu, nw, eh, nhh, tlo, thi);
    const float ah = std::fabs(thi), al = std::fabs(tlo);
    return (ah != ah || al != al) ? ah + al : (ah > al ? ah : al);
}

// stage 1's decision: maxndd = the largest -dd over the node's leaves.  false = no leaf of the node can be flagged.
MPCB_SCR_HD bool screen_stage1_pass(float tmax, float maxndd) { return !(scr_fma(tmax, tmax, maxndd) <= 0.f); }

}  // namespace mpcb
