// TEST HARNESS (not part of the product): compiles SHIPPED pieces of the CUDA library for the host with g++ --
// csrc/mpcb_exact.cuh (the float64 leaf evaluation whose results the library returns) and the invariant-divisor
// index decoding of csrc/mpcb_types.cuh, and the operator events of csrc/mpcb_events.cuh -- so that tests/test_shipped_code_on_host.py can check them against the
// reference's golden outputs and the oracle without a GPU.
#include <cmath>
#include <vector>

#include "mpcb_events.cuh"
#include "mpcb_exact.cuh"

// one operator event (kind 1 new_target(a, b), 2 turn_left(a), 3 turn_right(a)) on a pose: line[4] = x_t, y_t, x_0, y_0
extern "C" int mpcb_test_apply_event(int kind, double a, double b, double radius, double x, double y, double phi,
                                     int slow_before, double *line) {
    mpcb_loop_event e = {0, kind, a, b};
    int slow = slow_before;
    mpcb::apply_event(e, radius, x, y, phi, line, slow);
    return slow;
}

extern "C" void mpcb_test_fastdiv64(unsigned long long d, long long count, const unsigned long long *n,
                                    unsigned long long *q) {
    mpcb::FastDiv64 f;
    mpcb::fastdiv_init(f, d);
    for (long long i = 0; i < count; ++i) q[i] = f.div(n[i]);
}

extern "C" void mpcb_test_fastdiv32(unsigned d, long long count, const unsigned *n, unsigned *q) {
    mpcb::FastDiv32 f;
    mpcb::fastdiv32_init(f, d);
    for (long long i = 0; i < count; ++i) q[i] = f.div(n[i]);
}

// tables built as mpcb_set_grid builds them and solve parameters as prep_kernel builds them
struct HostSolve {
    std::vector<double4> tab, tab_slow;
    std::vector<double> vt, vt_slow;
    mpcb::LaunchArgs a;
    mpcb::SolveParams P;
};

static void host_solve_setup(HostSolve &hs, const double *v, int nv, const double *beta, int nb, double L, double delta_t,
                             int mode, int cost_kind, int H, const double *state, const double *target,
                             const double *origin, int slow, double v_min) {
    const int S = nv * nb;
    hs.tab.resize(S); hs.tab_slow.resize(S); hs.vt.resize(S); hs.vt_slow.resize(S);
    double vmin_grid = v[0];
    for (int i = 1; i < nv; ++i) vmin_grid = std::fmin(vmin_grid, v[i]);
    const double v_slow = vmin_grid > v_min ? vmin_grid : v_min;             // math_model_tree.py:312-316
    for (int iv = 0; iv < nv; ++iv)
        for (int ib = 0; ib < nb; ++ib) {
            const int c = iv * nb + ib;
            for (int variant = 0; variant < 2; ++variant) {
                const double vc = variant ? v_slow : v[iv];
                const double dphi = (vc / L) * std::tan(beta[ib]) * delta_t;   // math_model.py:77-78 x delta_t
                (variant ? hs.tab_slow : hs.tab)[c] = make_double4(std::cos(dphi), std::sin(dphi), vc * delta_t, dphi);
                (variant ? hs.vt_slow : hs.vt)[c] = vc;
            }
        }
    mpcb::LaunchArgs &a = hs.a;
    a = mpcb::LaunchArgs{};
    a.g.tab64 = hs.tab.data(); a.g.vtab = hs.vt.data(); a.g.tab64_slow = hs.tab_slow.data(); a.g.vtab_slow = hs.vt_slow.data();
    a.g.S = S; a.g.nb = nb; a.g.dt = delta_t;
    a.mode = mode; a.H = H; a.cost_kind = cost_kind;
    unsigned long long pw = 1;
    for (int k = H - 1; k >= 0; --k) {   // fd[k].d = S^(H-1-k), fd32 likewise where it fits, as fill_args (mpcb_api.cu)
        mpcb::fastdiv_init(a.fd[k], pw);
        if (pw < (1ULL << 32)) mpcb::fastdiv32_init(a.fd32[k], pw);
        if (mode == 0) pw *= (unsigned long long)S;
    }
    mpcb::SolveParams &P = hs.P;
    P = mpcb::SolveParams{};
    P.xs = state[0]; P.ys = state[1]; P.phi0 = state[2];
    P.xt = target[0]; P.yt = target[1];
    P.ox = origin[0]; P.oy = origin[1];
    P.theta = std::atan(P.xt / P.yt);
    P.lineA = P.yt - P.oy; P.lineB = P.xt - P.ox;
    P.lineC = P.xt * P.oy - P.yt * P.ox;
    P.line_norm = std::sqrt(P.lineA * P.lineA + P.lineB * P.lineB);
    P.flags = slow ? mpcb::kFlagSlow : 0;
}

// cost of leaf j of one solve (mode 0 FULL / 1 HELD), poses after each step and the first control, computed by
// mpcb::exact_cost
extern "C" double mpcb_test_exact_cost(const double *v, int nv, const double *beta, int nb, double L, double delta_t,
                                       int mode, int cost_kind, int H, const double *state, const double *target,
                                       const double *origin, long long j, double *traj, int *first_c, int slow,
                                       double v_min) {
    HostSolve hs;
    host_solve_setup(hs, v, nv, beta, nb, L, delta_t, mode, cost_kind, H, state, target, origin, slow, v_min);
    return mpcb::exact_cost(hs.a, hs.P, j, traj, first_c);
}

// the same leaves of a FULL tree the way the refinement scan evaluates them: the float64 pose of the leaf's depth-(H-1)
// node once (exact_node_pose, node digits decoded with the 32-bit dividers when node32 != 0), then one step per leaf
// (exact_child_cost).  out[i] must equal exact_cost(j[i]) bit for bit; digits_out[i * (H-1) + k] = the node's controls.
extern "C" void mpcb_test_exact_from_node(const double *v, int nv, const double *beta, int nb, double L, double delta_t,
                                          int cost_kind, int H, const double *state, const double *target,
                                          const double *origin, int slow, double v_min, int node32, long long count,
                                          const long long *j, double *out, double *out_whole, unsigned *digits_out,
                                          unsigned *parent_digits_out /* [count][H-2]: the controls of the node's parent */) {
    HostSolve hs;
    host_solve_setup(hs, v, nv, beta, nb, L, delta_t, 0, cost_kind, H, state, target, origin, slow, v_min);
    hs.a.node32 = node32;
    const unsigned long long S = (unsigned long long)(nv * nb);
    for (long long i = 0; i < count; ++i) {
        const unsigned long long p = (unsigned long long)j[i] / S;
        const unsigned c = (unsigned)((unsigned long long)j[i] - p * S);
        double x, y, phi;
        mpcb::exact_node_pose(hs.a, hs.P, p, x, y, phi);
        out[i] = mpcb::exact_child_cost(hs.a, hs.P, x, y, phi, c);
        out_whole[i] = mpcb::exact_cost(hs.a, hs.P, j[i], nullptr, nullptr);
        int k = 0;
        mpcb::node_digits(hs.a, p, [&](unsigned d) { digits_out[i * (H - 1) + k++] = d; });
        k = 0;
        mpcb::parent_digits(hs.a, p / S, [&](unsigned d) { parent_digits_out[i * (H - 2) + k++] = d; });
    }
}

// every leaf of one solve (mode 0 FULL: S^H leaves, 1 HELD: S), leaf order, by mpcb::exact_cost
extern "C" void mpcb_test_exact_costs(const double *v, int nv, const double *beta, int nb, double L, double delta_t,
                                      int mode, int cost_kind, int H, const double *state, const double *target,
                                      const double *origin, int slow, double v_min, long long count, double *out) {
    HostSolve hs;
    host_solve_setup(hs, v, nv, beta, nb, L, delta_t, mode, cost_kind, H, state, target, origin, slow, v_min);
    for (long long j = 0; j < count; ++j) out[j] = mpcb::exact_cost(hs.a, hs.P, j, nullptr, nullptr);
}
