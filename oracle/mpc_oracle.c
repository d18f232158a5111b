/* TEST INFRASTRUCTURE ONLY -- plain C (float64) restatement of the reference's MPC
 * inner loop, used where the numpy restatement (oracle/closed_form.py) is too slow:
 * parity tests on 1e7..1e9-leaf trees and bench.py's "closed-form CPU" baseline.
 * Never linked into, loaded by, or called from the product library.
 *
 * Follows (all into /root/reference):
 *   step   math_model.py:110-114  phi' = phi + dphi_c ; x' = x + v*cos(phi')*dt ; y' likewise
 *          (dphi_c = (v/L)*tan(beta)*dt is passed in as a table built by
 *           oracle/closed_form.control_tables so both oracles share bit-identical inputs)
 *   cost   math_model.py:48-58,82-86 (kind 0, "MM") / math_model_tree.py:56-66,82-87 (kind 1, "TREE")
 *   FULL   math_model.py:159-200: leaf j = sum_k i_k S^(H-1-k), first strict minimum wins
 *   HELD   math_model_tree.py:308-361: leaf k holds control k for H steps
 * Pinned against tests/golden (reference outputs) via tests/test_oracle_golden.py.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off -pthread; libgomp is not in this image,
 * so the first-control loop is spread over plain pthreads).
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <unistd.h>

typedef struct {
    const double *vv, *dphi;
    int S, H, cost_kind;
    double dt, xt, yt, x0, y0, theta, line_norm;
} ctx_t;

static double leaf_cost(const ctx_t *c, double x, double y, double phi)
{
    double dx = c->xt - x, dy = c->yt - y;
    double d = sqrt(dx * dx + dy * dy);
    double dl;
    if (x == c->x0 && y == c->y0)
        dl = 1000.0;
    else
        dl = fabs((c->yt - c->y0) * x - (c->xt - c->x0) * y + c->xt * c->y0 - c->yt * c->x0) / c->line_norm;
    if (c->cost_kind == 0) {
        double a = c->theta - phi;
        return 10000 * d + 10 * (a * a) + 100 * (dl * dl);
    }
    return 10000 * d + 10000 * (dl * dl);
}

static void dfs(const ctx_t *c, int depth, double x, double y, double phi, int64_t prefix,
                double *best, int64_t *best_idx)
{
    for (int i = 0; i < c->S; ++i) {
        double p = phi + c->dphi[i];
        double nx = x + c->vv[i] * cos(p) * c->dt;
        double ny = y + c->vv[i] * sin(p) * c->dt;
        int64_t j = prefix * c->S + i;
        if (depth + 1 == c->H) {
            double J = leaf_cost(c, nx, ny, p);
            if (J < *best) { *best = J; *best_idx = j; }
        } else {
            dfs(c, depth + 1, nx, ny, p, j, best, best_idx);
        }
    }
}


/* n work items: one per first control or -- split -- one per (first, second) control pair,
 * item k = (i0 - i0_begin) * S + i1, so that a range of a few first controls still spreads over every core.
 * Items in ascending order cover ascending, contiguous leaf-index ranges either way. */
typedef struct {
    const ctx_t *c; const double *state; int64_t i0_begin, n; int split; int64_t next; double *bc; int64_t *bi;
} job_t;

static int mpco_threads = 0;          /* 0 = all online cores */
void mpco_set_threads(int n) { mpco_threads = n; }
int mpco_get_threads(void) { return mpco_threads > 0 ? mpco_threads : (int)sysconf(_SC_NPROCESSORS_ONLN); }

static void *worker(void *arg)
{
    job_t *jb = (job_t *)arg;
    const ctx_t *c = jb->c;
    for (;;) {
        int64_t k = __atomic_fetch_add(&jb->next, 1, __ATOMIC_RELAXED);
        if (k >= jb->n) break;
        int64_t i0 = jb->i0_begin + (jb->split ? k / c->S : k);
        double best = INFINITY;
        int64_t idx = -1;
        double p = jb->state[2] + c->dphi[i0];
        double nx = jb->state[0] + c->vv[i0] * cos(p) * c->dt;
        double ny = jb->state[1] + c->vv[i0] * sin(p) * c->dt;
        if (c->H == 1) {
            double J = leaf_cost(c, nx, ny, p);
            if (J < best) { best = J; idx = i0; }
        } else if (jb->split) {           /* the second step as dfs() takes it */
            int i1 = (int)(k % c->S);
            double p1 = p + c->dphi[i1];
            double x1 = nx + c->vv[i1] * cos(p1) * c->dt;
            double y1 = ny + c->vv[i1] * sin(p1) * c->dt;
            int64_t j = i0 * c->S + i1;
            if (c->H == 2) {
                double J = leaf_cost(c, x1, y1, p1);
                if (J < best) { best = J; idx = j; }
            } else {
                dfs(c, 2, x1, y1, p1, j, &best, &idx);
            }
        } else {
            dfs(c, 1, nx, ny, p, i0, &best, &idx);
        }
        jb->bc[k] = best; jb->bi[k] = idx;
    }
    return NULL;
}

/* FULL tree restricted to first controls [i0_begin, i0_end). Returns the first
 * strict minimum (cost, global leaf index); index -1 if the range is empty or all NaN. */
int mpco_solve_full(const double *vv, const double *dphi, int S, int H, int cost_kind, double dt,
                    const double *state, const double *target, const double *origin, double theta,
                    int64_t i0_begin, int64_t i0_end, double *out_cost, int64_t *out_index)
{
    ctx_t c = {vv, dphi, S, H, cost_kind, dt, target[0], target[1], origin[0], origin[1], theta, 0.0};
    c.line_norm = sqrt((c.yt - c.y0) * (c.yt - c.y0) + (c.xt - c.x0) * (c.xt - c.x0));
    int64_t n = i0_end - i0_begin;
    if (n <= 0) { *out_cost = INFINITY; *out_index = -1; return 0; }
    int nt = mpco_threads > 0 ? mpco_threads : (int)sysconf(_SC_NPROCESSORS_ONLN);
    const int split = H >= 2 && n < 4 * (int64_t)nt;   /* few first controls: hand out (i0, i1) pairs */
    if (split) n *= S;
    double *bc = (double *)malloc(sizeof(double) * n);
    int64_t *bi = (int64_t *)malloc(sizeof(int64_t) * n);
    job_t job = {&c, state, i0_begin, n, split, 0, bc, bi};
    if (nt > n) nt = (int)n;
    if (nt < 1) nt = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * nt);
    for (int t = 1; t < nt; ++t) pthread_create(&th[t], NULL, worker, &job);
    worker(&job);
    for (int t = 1; t < nt; ++t) pthread_join(th[t], NULL);
    free(th);
    double best = INFINITY; int64_t idx = -1;
    for (int64_t k = 0; k < n; ++k)
        if (bc[k] < best) { best = bc[k]; idx = bi[k]; }   /* ascending items, strict: lowest index wins ties */
    free(bc); free(bi);
    *out_cost = best; *out_index = idx;
    return 0;
}

/* HELD: S candidates, candidate k repeats control k for H steps. Optionally writes all S costs. */
int mpco_solve_held(const double *vv, const double *dphi, int S, int H, int cost_kind, double dt,
                    const double *state, const double *target, const double *origin, double theta,
                    double *out_cost, int64_t *out_index, double *all_costs)
{
    ctx_t c = {vv, dphi, S, H, cost_kind, dt, target[0], target[1], origin[0], origin[1], theta, 0.0};
    c.line_norm = sqrt((c.yt - c.y0) * (c.yt - c.y0) + (c.xt - c.x0) * (c.xt - c.x0));
    double best = INFINITY; int64_t idx = -1;
    for (int k = 0; k < S; ++k) {
        double x = state[0], y = state[1], p = state[2];
        for (int h = 0; h < H; ++h) {
            p = p + dphi[k];
            x = x + vv[k] * cos(p) * dt;
            y = y + vv[k] * sin(p) * dt;
        }
        double J = leaf_cost(&c, x, y, p);
        if (all_costs) all_costs[k] = J;
        if (J < best) { best = J; idx = k; }
    }
    *out_cost = best; *out_index = idx;
    return 0;
}

/* Every leaf cost of a small FULL tree, enumeration order (S^H doubles). */
static void dfs_all(const ctx_t *c, int depth, double x, double y, double phi, int64_t prefix, double *out)
{
    for (int i = 0; i < c->S; ++i) {
        double p = phi + c->dphi[i];
        double nx = x + c->vv[i] * cos(p) * c->dt;
        double ny = y + c->vv[i] * sin(p) * c->dt;
        int64_t j = prefix * c->S + i;
        if (depth + 1 == c->H) out[j] = leaf_cost(c, nx, ny, p);
        else dfs_all(c, depth + 1, nx, ny, p, j, out);
    }
}

int mpco_full_leaf_costs(const double *vv, const double *dphi, int S, int H, int cost_kind, double dt,
                         const double *state, const double *target, const double *origin, double theta,
                         double *out)
{
    ctx_t c = {vv, dphi, S, H, cost_kind, dt, target[0], target[1], origin[0], origin[1], theta, 0.0};
    c.line_norm = sqrt((c.yt - c.y0) * (c.yt - c.y0) + (c.xt - c.x0) * (c.xt - c.x0));
    dfs_all(&c, 0, state[0], state[1], state[2], 0, out);
    return 0;
}
