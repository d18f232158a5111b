// TEST HARNESS (not part of the product): compiles the SHIPPED stage-1 bound of the two-stage screen,
// diplomjourney_b200/csrc/mpcb_screen.cuh, for the host with g++, next to a replay of the fp32 arithmetic of the
// screen loop (prefix_screen_loop_rows / prefix_dist_loop_rows in mpcb_kernels.cu), so that
// tests/test_screen_stage1_on_host.py can check the bound against every leaf of small trees.
#include <cfloat>
#include <cmath>
#include <cstring>

#include "mpcb_screen.cuh"

namespace {

constexpr float kWd2f = 1.0e8f;

// one node's registers as the kernel holds them: u2s, w2s, D2s, nu, nw, eh, nhh
struct Node {
    float u2s, w2s, D2s, nu, nw, eh, nhh;
};

Node node_at(const float *regs, long long i) {
    const float *r = regs + 7 * i;
    return Node{r[0], r[1], r[2], r[3], r[4], r[5], r[6]};
}

// the leaf's terms with the operands and operations of the kernel's loops (-dd, q, gg, t, fma(t, t, -dd))
struct Leaf {
    float ndd, q, gg, t, df;
};

Leaf leaf_terms(const float *e, const Node &p, float cn, bool head) {
    Leaf l;
    const float DV = std::fma(-kWd2f, e[2], -p.D2s);
    l.ndd = std::fma(-p.u2s, e[0], std::fma(-p.w2s, e[1], DV));
    l.q = std::fma(p.nu, e[0], std::fma(p.nw, e[1], p.eh));
    l.gg = e[3] + p.nhh;
    l.t = std::fma(-l.q, l.q, cn);
    if (head) l.t = std::fma(-l.gg, l.gg, l.t);
    l.df = std::fma(l.t, l.t, l.ndd);
    return l;
}

bool flagged_with_positive_t(const float *tab, int S, const Node &p, float cn, bool head) {
    for (int c = 0; c < S; ++c) {
        const Leaf l = leaf_terms(tab + 4 * c, p, cn, head);
        if (l.t > 0.f && l.df > 0.f) return true;
    }
    return false;
}

}  // namespace

// Per node i (n nodes, tab = S controls x {a, b, r, g} in fp32, box = amin, amax, bmin, bmax, gmin, gmax; tshrink: the
// stage-1 T is lowered by that many ulps before the decision -- 0 is the shipped decision), out[16 i + ...]:
//   0 the stage-2 maximum of fma(t, t, -dd) over the leaves, 1 stage 1's maximum of -dd, 2 T, 3 stage 1 passes (0 / 1),
//   4 / 5 min / max of t over the leaves, 6 / 7 the bound's tlo / thi, 8 / 9 min / max q, 10 / 11 the bound's q range,
//   12 / 13 min / max gg, 14 / 15 the bound's gg range
extern "C" void mpcb_test_screen(int S, const float *tab, const float *box6, int head, long long n, const float *regs,
                                 const float *cn, int tshrink, float *out) {
    const mpcb::ScreenBox bx{box6[0], box6[1], box6[2], box6[3], box6[4], box6[5]};
    for (long long i = 0; i < n; ++i) {
        const Node p = node_at(regs, i);
        float mx = -INFINITY, mndd = -INFINITY, tmin = INFINITY, tmax_ = -INFINITY;
        float qmin = INFINITY, qmax = -INFINITY, gmin = INFINITY, gmax = -INFINITY;
        for (int c = 0; c < S; ++c) {
            const Leaf l = leaf_terms(tab + 4 * c, p, cn[i], head != 0);
            mx = std::fmax(mx, l.df); mndd = std::fmax(mndd, l.ndd);
            tmin = std::fmin(tmin, l.t); tmax_ = std::fmax(tmax_, l.t);
            qmin = std::fmin(qmin, l.q); qmax = std::fmax(qmax, l.q);
            gmin = std::fmin(gmin, l.gg); gmax = std::fmax(gmax, l.gg);
        }
        float T = mpcb::screen_stage1_tmax(bx, head != 0, cn[i], p.nu, p.nw, p.eh, p.nhh);
        for (int k = 0; k < tshrink; ++k) T = std::nextafter(T, 0.f);
        float *o = out + 16 * i;
        o[0] = mx; o[1] = mndd; o[2] = T; o[3] = mpcb::screen_stage1_pass(T, mndd) ? 1.f : 0.f;
        o[4] = tmin; o[5] = tmax_;
        mpcb::screen_t_range(bx, head != 0, cn[i], p.nu, p.nw, p.eh, p.nhh, o[6], o[7]);
        o[8] = qmin; o[9] = qmax;
        mpcb::screen_q_range(bx, p.nu, p.nw, p.eh, o[10], o[11]);
        o[12] = gmin; o[13] = gmax;
        mpcb::screen_g_range(bx, p.nhh, o[14], o[15]);
    }
}

// Per node: the smallest cn >= 0 at which the screen flags the node through a leaf with t > 0 (bisection over the
// ordered fp32 bit patterns; the predicate does not decrease with cn), NaN if none up to FLT_MAX.
extern "C" void mpcb_test_knife_edge_cn(int S, const float *tab, int head, long long n, const float *regs, float *out) {
    for (long long i = 0; i < n; ++i) {
        const Node p = node_at(regs, i);
        if (!flagged_with_positive_t(tab, S, p, FLT_MAX, head != 0)) { out[i] = NAN; continue; }
        unsigned lo = 0, hi = 0x7f7fffffu;                  // flagged at hi, maybe at lo
        float f;
        std::memcpy(&f, &lo, 4);
        if (flagged_with_positive_t(tab, S, p, f, head != 0)) { out[i] = f; continue; }
        while (hi - lo > 1) {
            const unsigned mid = lo + (hi - lo) / 2;
            std::memcpy(&f, &mid, 4);
            if (flagged_with_positive_t(tab, S, p, f, head != 0)) hi = mid; else lo = mid;
        }
        std::memcpy(&out[i], &hi, 4);
    }
}
