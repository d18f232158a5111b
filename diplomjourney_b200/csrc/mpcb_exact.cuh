// mpcb_exact.cuh -- the float64 evaluation of a leaf by the reference's own formula and operation order: what the
// refinement pass and the final re-roll of the winner compute, i.e. the numbers the library returns.
//
// Plain host/device functions, so that the CPU test-suite can compile exactly this code with g++ (-ffp-contract=off) and
// compare it with the reference's golden outputs (tests/test_shipped_code_on_host.py); mpcb_kernels.cu includes it as is.
#pragma once
#include <cmath>

#include "mpcb_types.cuh"

namespace mpcb {

// the controls i_0 .. i_{H-2} of depth-(H-1) node p, first step first: step(i) once per digit.  fd[k + 1].d = S^(H-2-k), so
// the last digit is what is left (no division by 1), and indices below 2^32 take the 5-instruction 32-bit dividers
template <typename F>
MPCB_HD void node_digits(const LaunchArgs &a, unsigned long long p, F &&step) {
    const int D = a.H - 1;
    if (D <= 0) return;
    if (a.node32) {
        unsigned rem = (unsigned)p;
        for (int k = 0; k + 1 < D; ++k) {
            const unsigned i = a.fd32[k + 1].div(rem);
            rem -= i * a.fd32[k + 1].d;
            step(i);
        }
        step(rem);
    } else {
        unsigned long long rem = p;
        for (int k = 0; k + 1 < D; ++k) {
            const unsigned long long i = a.fd[k + 1].div(rem);
            rem -= i * a.fd[k + 1].d;
            step((unsigned)i);
        }
        step((unsigned)rem);
    }
}

// ... and the controls i_0 .. i_{H-3} of depth-(H-2) node q (fd[k + 2].d = S^(H-3-k))
template <typename F>
MPCB_HD void parent_digits(const LaunchArgs &a, unsigned long long q, F &&step) {
    const int D = a.H - 2;
    if (D <= 0) return;
    if (a.node32) {
        unsigned rem = (unsigned)q;
        for (int k = 0; k + 1 < D; ++k) {
            const unsigned i = a.fd32[k + 2].div(rem);
            rem -= i * a.fd32[k + 2].d;
            step(i);
        }
        step(rem);
    } else {
        unsigned long long rem = q;
        for (int k = 0; k + 1 < D; ++k) {
            const unsigned long long i = a.fd[k + 2].div(rem);
            rem -= i * a.fd[k + 2].d;
            step((unsigned)i);
        }
        step((unsigned)rem);
    }
}

// ---- float64 evaluation by the reference's own formula and operation order
// (iteration_of_predict math_model.py:110-114, control_criterion :82-86 / tree :82-87)
MPCB_HD void exact_step(const LaunchArgs &a, const double4 *tab, const double *vt,
                                           unsigned long long c, double &x, double &y, double &phi) {
    const double dphi = ro_load(&tab[c].w);
    const double v = ro_load(&vt[c]);
    phi = dadd(phi, dphi);
    double sn, cs;
#ifdef __CUDA_ARCH__
    sincos(phi, &sn, &cs);
#else
    sn = std::sin(phi); cs = std::cos(phi);
#endif
    x = dadd(x, dmul(dmul(v, cs), a.g.dt));
    y = dadd(y, dmul(dmul(v, sn), a.g.dt));
}

MPCB_HD double exact_terminal(const LaunchArgs &a, const SolveParams &P, double x, double y,
                                                 double phi) {
    double dx = P.xt - x, dy = P.yt - y;
    double d = dsqrt(dadd(dmul(dx, dx), dmul(dy, dy)));
    double dl;
    if (x == P.ox && y == P.oy) dl = 1000.0;
    else
        dl = fabs(dadd(dadd(dadd(dmul(P.lineA, x), -dmul(P.lineB, y)), dmul(P.xt, P.oy)), -dmul(P.yt, P.ox))) /
             P.line_norm;     // ((A x - B y) + x_t y_0) - y_t x_0, left to right as the reference
    double dl2 = dmul(dl, dl);
    if (a.cost_kind == 0) {
        double ang = P.theta - phi;
        return dadd(dadd(dmul(10000.0, d), dmul(10.0, dmul(ang, ang))),
                         dmul(100.0, dl2));
    }
    return dadd(dmul(10000.0, d), dmul(10000.0, dl2));
}

// cost of leaf j (whole walk); optionally returns the poses after each step and the first control
MPCB_HD_NOINLINE double exact_cost(const LaunchArgs &a, const SolveParams &P, long long j,
                                          double *traj /* [H][3] or null */, int *first_c) {
    const bool slow = (P.flags & kFlagSlow) != 0;
    const double4 *tab = slow ? a.g.tab64_slow : a.g.tab64;
    const double *vt = slow ? a.g.vtab_slow : a.g.vtab;
    double x = P.xs, y = P.ys, phi = P.phi0;
    unsigned long long rem = (unsigned long long)j;
    for (int k = 0; k < a.H; ++k) {
        unsigned long long c;
        if (a.mode == 1) c = (unsigned long long)j;
        else { c = a.fd[k].div(rem); rem -= c * a.fd[k].d; }
        if (k == 0 && first_c) *first_c = (int)c;
        exact_step(a, tab, vt, c, x, y, phi);
        if (traj) { traj[3 * k] = x; traj[3 * k + 1] = y; traj[3 * k + 2] = phi; }
    }
    return exact_terminal(a, P, x, y, phi);
}

// float64 pose of depth-(H-1) node p by the reference's own steps: exactly what exact_cost computes on the way to any
// leaf below it, so  exact_child_cost(pose, c) == exact_cost(p * S + c)  bit for bit (FULL trees)
// (both out of line, like exact_cost: inlined, their double-precision sincos took the scan loop's registers)
MPCB_HD_NOINLINE void exact_node_pose(const LaunchArgs &a, const SolveParams &P, unsigned long long p, double &x,
                                             double &y, double &phi) {
    const bool slow = (P.flags & kFlagSlow) != 0;
    const double4 *tab = slow ? a.g.tab64_slow : a.g.tab64;
    const double *vt = slow ? a.g.vtab_slow : a.g.vtab;
    x = P.xs; y = P.ys; phi = P.phi0;
    node_digits(a, p, [&](unsigned i) { exact_step(a, tab, vt, i, x, y, phi); });
}
MPCB_HD_NOINLINE double exact_child_cost(const LaunchArgs &a, const SolveParams &P, double x, double y, double phi,
                                                unsigned c) {
    const bool slow = (P.flags & kFlagSlow) != 0;
    exact_step(a, slow ? a.g.tab64_slow : a.g.tab64, slow ? a.g.vtab_slow : a.g.vtab, c, x, y, phi);
    return exact_terminal(a, P, x, y, phi);
}

}  // namespace mpcb
