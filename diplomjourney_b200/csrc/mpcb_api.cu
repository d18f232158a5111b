// mpcb_api.cu -- host side of the C ABI declared in include/mpcb200.h.
//
// One handle = one device + one stream + growable device scratch.  A solve enqueues
//   prep -> pass 1 (partial minima) -> reduce+compact -> pass 2 (float64 refinement) -> finalize
// on the handle's stream; the "_host" entry points add the H2D/D2H copies and a sync.
#include "../../include/mpcb200.h"
#include "mpcb_types.cuh"
#include "mpcb_bounds.cuh"
#include "mpcb_handle.cuh"
#include "mpcb_noise.cuh"
#include "mpcb_pcg64.cuh"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace mpcb {
cudaError_t launch_prep(cudaStream_t, long long, const double *, const double *, const double *, const double *,
                        const uint8_t *, int, int, int, double, double, double, SolveParams *);
cudaError_t launch_pass(cudaStream_t, const LaunchArgs &, const RowPairs &, int pass, bool prefix, int sms);
cudaError_t launch_reduce_compact(cudaStream_t, const LaunchArgs &, double *, unsigned *, unsigned *, int sms);
cudaError_t launch_reduce_compact_wide(cudaStream_t, const LaunchArgs &, double *, unsigned *, unsigned *, void *scratch,
                                       int sms, int *launches);
cudaError_t launch_probe(cudaStream_t, const LaunchArgs &, int sms);
cudaError_t launch_tilecut(cudaStream_t, const LaunchArgs &, unsigned long long g_begin, unsigned long long g_end,
                           unsigned long long *list, unsigned *count, unsigned long long list_cap);
cudaError_t launch_frontier_expand(cudaStream_t, const LaunchArgs &, int k, const unsigned long long *src,
                                   const unsigned *src_count, unsigned long long *dst, unsigned *dst_count,
                                   unsigned *overflow, int sms);
cudaError_t launch_tilewalk_fallback(cudaStream_t, const LaunchArgs &, unsigned long long all_tiles, int sms);
cudaError_t launch_cand_resolve(cudaStream_t, const LaunchArgs &, int sms);
cudaError_t launch_refine_scan(cudaStream_t, const LaunchArgs &, int sms);
cudaError_t launch_finalize(cudaStream_t, const LaunchArgs &, double *, long long *, double *, double *);
cudaError_t launch_dump(cudaStream_t, const LaunchArgs &, bool prefix, double *jrel, int sms);
cudaError_t launch_held_loop(cudaStream_t, const LoopArgs &, int sms);
cudaError_t launch_rng_seed(cudaStream_t, long long N, const unsigned *keys, int key_len, unsigned *rng_state);
cudaError_t launch_pcg64_seed(cudaStream_t, long long N, const unsigned *entropy, int ent_len, int ent_stride,
                              const unsigned *spawn, int spawn_len, unsigned long long *pcg_state);
cudaError_t launch_held_small(cudaStream_t, const SmallArgs &);
cudaError_t launch_full_apply(cudaStream_t, const FullLoopArgs &);
cudaError_t launch_full_loop_init(cudaStream_t, const FullLoopArgs &, const double *init, const double *first_threshold);
cudaError_t launch_full_loop_gate(cudaStream_t, cudaGraphConditionalHandle, int *ctl, int max_ticks, int advance);
cudaError_t launch_held_windows(cudaStream_t, const WindowArgs &, int sms);
cudaError_t launch_held_ctrl_init(cudaStream_t, long long N, const double *init, const double *target,
                                  const double *origin, const double *first_threshold, const int *slow_steps,
                                  mpcb_held_ctrl *ctrl);
cudaError_t launch_held_ctrl_step(cudaStream_t, const HeldCtrlArgs &, int sms);
cudaError_t launch_split_ub_min(cudaStream_t, const LaunchArgs &, const unsigned long long *all, int nranks);
cudaError_t launch_split_pack(cudaStream_t, const LaunchArgs &, SplitRec *mine);
cudaError_t launch_split_pick(cudaStream_t, const LaunchArgs &, const SplitRec *all, int nranks);
bool nccl_available();
int nccl_comm_info(void *comm, int *nranks, int *rank);
int nccl_allgather_bytes(void *comm, const void *send, void *recv, size_t bytes, cudaStream_t st);
}  // namespace mpcb

using namespace mpcb;

namespace {

int fail(mpcb_handle *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(h, MPCB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                       \
    } while (0)

// S^H as unsigned 64-bit with overflow check against int64
bool pow_checked(unsigned long long S, int H, unsigned long long &out) {
    unsigned __int128 r = 1;
    for (int i = 0; i < H; ++i) {
        r *= S;
        if (r > (unsigned __int128)INT64_MAX) return false;
    }
    out = (unsigned long long)r;
    return true;
}

struct Plan {
    bool prefix;
    unsigned long long u_begin, u_end, leaves_per_solve;
    long long i0_begin = 0, i0_end = 0;
};

int make_plan(mpcb_handle *h, int mode, int H, long long N, long long i0_begin, long long i0_end, int algo_req,
              Plan &pl) {
    const unsigned long long S = (unsigned long long)h->g.S;
    if (mode == MPCB_MODE_HELD) {
        pl.prefix = false;
        pl.u_begin = 0; pl.u_end = S; pl.leaves_per_solve = S;
        return MPCB_OK;
    }
    unsigned long long leaves = 0, sub = 1;
    if (!pow_checked(S, H, leaves)) return fail(h, MPCB_ERR_TOO_LARGE, "S^H = %llu^%d exceeds int64", S, H);
    pow_checked(S, H - 1, sub);
    if (i0_end < 0) { i0_begin = 0; i0_end = (long long)S; }
    if (i0_begin < 0 || i0_end > (long long)S || i0_begin > i0_end)
        return fail(h, MPCB_ERR_INVALID, "bad first-control range [%lld,%lld) for S=%llu", i0_begin, i0_end, S);
    int algo = algo_req == MPCB_ALGO_AUTO ? h->algo : algo_req;
    const unsigned long long parents = H >= 2 ? sub : 0;   // S^(H-1) depth-(H-1) nodes
    if (algo == MPCB_ALGO_AUTO)
        algo = (H >= 2 && (unsigned __int128)parents * (unsigned long long)N >= 32768) ? MPCB_ALGO_PREFIX
                                                                                       : MPCB_ALGO_LEAFWALK;
    if (H < 2) algo = MPCB_ALGO_LEAFWALK;
    pl.prefix = algo == MPCB_ALGO_PREFIX;
    if (pl.prefix) {
        unsigned long long per_i0 = sub / S;   // S^(H-2) depth-(H-1) nodes below one first control
        pl.u_begin = (unsigned long long)i0_begin * per_i0;
        pl.u_end = (unsigned long long)i0_end * per_i0;
    } else {
        pl.u_begin = (unsigned long long)i0_begin * sub;
        pl.u_end = (unsigned long long)i0_end * sub;
    }
    pl.leaves_per_solve = (unsigned long long)(i0_end - i0_begin) * sub;
    pl.i0_begin = i0_begin; pl.i0_end = i0_end;
    return MPCB_OK;
}

void fill_args(mpcb_handle *h, LaunchArgs &a, int mode, int cost_kind, int H, long long N, const Plan &pl) {
    memset(&a, 0, sizeof a);
    a.g = h->g;
    a.mode = mode; a.H = H; a.cost_kind = cost_kind; a.refine = h->refine;
    a.dump_direct = h->dump_direct; a.npt = h->npt;
    a.N = N;
    unsigned long long S = (unsigned long long)h->g.S, pw = 1;
    a.idx32 = (!pl.prefix && pl.u_end < (1ULL << 32)) ? 1 : 0;
    // prefix algorithm: units are depth-(H-1) nodes, decoded with fd[1..H-1]; 32-bit dividers when every node index fits
    a.node32 = (pl.prefix && pl.u_end < (1ULL << 32)) ? 1 : 0;
    for (int k = H - 1; k >= 0; --k) {   // fd[k].d = S^(H-1-k)
        fastdiv_init(a.fd[k], pw);
        if ((a.idx32 || (a.node32 && k >= 1)) && pw < (1ULL << 32)) fastdiv32_init(a.fd32[k], pw);
        else if (a.node32 && k >= 1) a.node32 = 0;
        if (mode == MPCB_MODE_FULL) pw *= S;
    }
    a.u_begin = pl.u_begin; a.u_end = pl.u_end;
    a.i0_begin = (int)pl.i0_begin; a.i0_end = (int)pl.i0_end;
    {   // digits of kThreads in base S over H positions (leafwalk's incremental index decode)
        unsigned long long r = kThreads;
        for (int k = H - 1; k >= 0; --k) { a.step_digits[k] = mode == MPCB_MODE_FULL ? (unsigned)(r % S) : 0u; r = mode == MPCB_MODE_FULL ? r / S : 0; }
    }
    bounds_set_heading_ranges(a, h->g.dphimax);   // heading range after i+1 steps, for the pruning bounds
    a.tile_units = pl.prefix ? kThreads : kThreads * kLeafPerThread;
    a.lw_smem = (!pl.prefix && mode == MPCB_MODE_FULL && h->g.S <= 4096) ? 1 : 0;
}

}  // namespace

static int ensure_tables(mpcb_handle *h) {
    if (h->tables_ready) return MPCB_OK;
    const double *v = h->hv.data(), *beta = h->hb.data();
    const int nv = (int)h->hv.size(), nb = (int)h->hb.size();
    const double L = h->L, delta_t = h->delta_t, v_min = h->v_min;
    CK(cudaSetDevice(h->device));
    const int S = nv * nb;
    std::vector<double4> t64(S), t64s(S);
    std::vector<double> vt(S), vts(S);
    std::vector<float4> l32(S);
    std::vector<float2> c32(S), c32s(S);
    double vmin_grid = v[0];
    for (int i = 1; i < nv; ++i) vmin_grid = std::min(vmin_grid, v[i]);
    const double v_slow = vmin_grid > v_min ? vmin_grid : v_min;   // math_model_tree.py:312-316
    double smax = 0, dphimax = 0, smin = INFINITY;
    for (int iv = 0; iv < nv; ++iv)
        for (int ib = 0; ib < nb; ++ib) {
            const int c = iv * nb + ib;
            for (int variant = 0; variant < 2; ++variant) {
                const double vc = variant ? v_slow : v[iv];
                const double dphi = (vc / L) * std::tan(beta[ib]) * delta_t;   // math_model.py:77-78 x delta_t
                const double s = vc * delta_t;
                const double cd = std::cos(dphi), sd = std::sin(dphi);
                smax = std::max(smax, std::fabs(s));
                smin = std::min(smin, s);
                dphimax = std::max(dphimax, std::fabs(dphi));
                if (variant == 0) {
                    t64[c] = make_double4(cd, sd, s, dphi);
                    vt[c] = vc;
                    l32[c] = make_float4((float)(s * cd), (float)(s * sd), (float)(s * s),
                                         (float)(3.16227766016837952 * dphi));
                    c32[c] = make_float2((float)dphi, (float)s);
                } else {
                    t64s[c] = make_double4(cd, sd, s, dphi);
                    vts[c] = vc;
                    c32s[c] = make_float2((float)dphi, (float)s);
                }
            }
        }
    std::vector<float4> t32(S);
    for (int c = 0; c < S; ++c) t32[c] = make_float4((float)t64[c].x, (float)t64[c].y, (float)t64[c].z, (float)t64[c].w);
    CK(h->tab32.ensure(sizeof(float4) * S));
    CK(h->tab64.ensure(sizeof(double4) * S)); CK(h->tab64_slow.ensure(sizeof(double4) * S));
    CK(h->vtab.ensure(sizeof(double) * S)); CK(h->vtab_slow.ensure(sizeof(double) * S));
    CK(h->beta.ensure(sizeof(double) * nb));
    // pair table for the packed pass-1 loop; chunk boundaries (kLeafChunk, even) keep pairs intact
    const int npairs = (S + 1) / 2;
    std::vector<float4> l32p(2 * (size_t)npairs);
    for (int m = 0; m < npairs; ++m) {
        const float4 x = l32[2 * m], y = l32[std::min(2 * m + 1, S - 1)];
        l32p[2 * m] = make_float4(x.x, y.x, x.y, y.y);
        l32p[2 * m + 1] = make_float4(x.z, y.z, x.w, y.w);
    }
    // the same pairs by speed row, when the whole table fits one shared-memory chunk (screened pass 1: K r + D2 once per row)
    const int ppr = (nb + 1) / 2;
    const bool rows_fit = 2LL * nv * ppr <= kLeafChunk;
    std::vector<float4> l32r(rows_fit ? 2 * (size_t)nv * ppr : 0);
    if (rows_fit)
        for (int iv = 0; iv < nv; ++iv)
            for (int m = 0; m < ppr; ++m) {
                const float4 x = l32[iv * nb + 2 * m], y = l32[iv * nb + std::min(2 * m + 1, nb - 1)];
                l32r[2 * ((size_t)iv * ppr + m)] = make_float4(x.x, y.x, x.y, y.y);
                l32r[2 * ((size_t)iv * ppr + m) + 1] = make_float4(x.z, y.z, x.w, y.w);
                h->row_ab.ab[iv * ppr + m] = l32r[2 * ((size_t)iv * ppr + m)];
            }
    CK(h->leaf32r.ensure(sizeof(float4) * std::max<size_t>(l32r.size(), 1)));
    CK(h->leaf32.ensure(sizeof(float4) * S));
    CK(h->leaf32p.ensure(sizeof(float4) * 2 * npairs));
    CK(h->ctl32.ensure(sizeof(float2) * S)); CK(h->ctl32_slow.ensure(sizeof(float2) * S));
    // pageable sources: cudaMemcpyAsync stages them before returning, so the vectors may die here;
    // ordering against earlier solves on the stream is preserved
    CK(cudaMemcpyAsync(h->tab64.p, t64.data(), sizeof(double4) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->tab32.p, t32.data(), sizeof(float4) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->tab64_slow.p, t64s.data(), sizeof(double4) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->vtab.p, vt.data(), sizeof(double) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->vtab_slow.p, vts.data(), sizeof(double) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->beta.p, beta, sizeof(double) * nb, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->leaf32.p, l32.data(), sizeof(float4) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->leaf32p.p, l32p.data(), sizeof(float4) * 2 * npairs, cudaMemcpyHostToDevice, h->stream));
    if (rows_fit) CK(cudaMemcpyAsync(h->leaf32r.p, l32r.data(), sizeof(float4) * l32r.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->ctl32.p, c32.data(), sizeof(float2) * S, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->ctl32_slow.p, c32s.data(), sizeof(float2) * S, cudaMemcpyHostToDevice, h->stream));
    GridTables &g = h->g;
    g.tab64 = h->tab64.as<double4>(); g.vtab = h->vtab.as<double>();
    g.tab32 = h->tab32.as<float4>();
    g.tab64_slow = h->tab64_slow.as<double4>(); g.vtab_slow = h->vtab_slow.as<double>();
    g.beta = h->beta.as<double>();
    g.leaf32 = h->leaf32.as<float4>();
    g.leaf32p = h->leaf32p.as<float4>();
    g.leaf32r = rows_fit ? h->leaf32r.as<float4>() : nullptr;
    g.nv = nv; g.ppr = rows_fit ? ppr : 0;
    g.ctl32 = h->ctl32.as<float2>(); g.ctl32_slow = h->ctl32_slow.as<float2>();
    g.S = S; g.nb = nb; g.dt = delta_t; g.smax = smax; g.dphimax = dphimax; g.smin = smin;
    g.sbox = ScreenBox{l32[0].x, l32[0].x, l32[0].y, l32[0].y, l32[0].w, l32[0].w};
    for (int c = 1; c < S; ++c) {
        g.sbox.amin = std::min(g.sbox.amin, l32[c].x); g.sbox.amax = std::max(g.sbox.amax, l32[c].x);
        g.sbox.bmin = std::min(g.sbox.bmin, l32[c].y); g.sbox.bmax = std::max(g.sbox.bmax, l32[c].y);
        g.sbox.gmin = std::min(g.sbox.gmin, l32[c].w); g.sbox.gmax = std::max(g.sbox.gmax, l32[c].w);
    }
    h->tables_ready = true;
    return MPCB_OK;
}


extern "C" {

static void retire_loop_graphs(mpcb_handle *h, bool all);

int mpcb_version(void) { return 100; }

int mpcb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int mpcb_create(int device_ordinal, mpcb_handle **out) {
    if (!out) return MPCB_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return MPCB_ERR_NO_DEVICE;
    if (device_ordinal < 0 || device_ordinal >= n) return MPCB_ERR_INVALID;
    mpcb_handle *h = new mpcb_handle_s();
    h->device = device_ordinal;
    if (cudaSetDevice(device_ordinal) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return MPCB_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, device_ordinal);
    *out = h;
    return MPCB_OK;
}

int mpcb_destroy(mpcb_handle *h) {
    if (!h) return MPCB_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (DevBuf *b : {&h->tab64, &h->tab32, &h->vtab, &h->tab64_slow, &h->vtab_slow, &h->beta, &h->leaf32, &h->leaf32p, &h->leaf32r, &h->ctl32,
                      &h->ctl32_slow, &h->sp, &h->segmin, &h->worklist, &h->misc, &h->tau, &h->bestJ, &h->bestIdx,
                      &h->lock, &h->ub, &h->tile_list, &h->reduce_scratch, &h->in_state, &h->in_target, &h->in_origin, &h->in_thr, &h->in_flags, &h->out_cost,
                      &h->out_index, &h->out_traj, &h->out_ctl, &h->dump_rec, &h->dump_j, &h->loop_log, &h->loop_ticks,
                      &h->loop_status, &h->loop_events, &h->loop_final, &h->loop_rng, &h->loop_keys, &h->small_in, &h->small_out, &h->fl_last, &h->fl_k, &h->fl_have, &h->fl_flags,
                      &h->fl_count, &h->fl_state, &h->fl_thr, &h->trace_pred, &h->trace_ctl, &h->trace_cost, &h->fl_traj, &h->nccl_scratch, &h->cand, &h->cand_J, &h->cand_sel, &h->node_list})
        b->release();
    retire_loop_graphs(h, true);
    if (h->fl_exec) cudaGraphExecDestroy(h->fl_exec);
    if (h->pin_in) cudaFreeHost(h->pin_in);
    if (h->pin_out) cudaFreeHost(h->pin_out);
    cudaStreamDestroy(h->stream);
    delete h;
    return MPCB_OK;
}

const char *mpcb_last_error(const mpcb_handle *h) { return h ? h->err.c_str() : "null handle"; }
void *mpcb_stream(mpcb_handle *h) { return h ? (void *)h->stream : nullptr; }

int mpcb_sync(mpcb_handle *h) {
    if (!h) return MPCB_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return MPCB_OK;
}

int mpcb_set_option(mpcb_handle *h, const char *name, double value) {
    if (!h || !name) return MPCB_ERR_INVALID;
    ++h->epoch;
    if (!strcmp(name, "tol_scale")) h->tol_scale = value;
    else if (!strcmp(name, "algo")) h->algo = (int)value;
    else if (!strcmp(name, "refine")) h->refine = value != 0.0;
    else if (!strcmp(name, "small_path")) h->small_path = value != 0.0;
    else if (!strcmp(name, "zero_copy")) h->zero_copy = value != 0.0;
    else if (!strcmp(name, "candidate_list")) {
        if (value == -1.0) { h->cand_cap = 1u << 20; h->cand_auto = true; return MPCB_OK; }
        if (!(value >= 0.0 && value <= (double)(1u << 26))) return fail(h, MPCB_ERR_INVALID, "candidate_list out of range [0, 2^26] (or -1)");
        h->cand_cap = (unsigned)value; h->cand_auto = false;
    }
    else if (!strcmp(name, "node_list")) {
        if (!(value >= 0.0 && value <= (double)(1u << 24))) return fail(h, MPCB_ERR_INVALID, "node_list out of range [0, 2^24]");
        h->node_cap = (unsigned)value;
    }
    else if (!strcmp(name, "prune")) h->prune = value != 0.0;
    else if (!strcmp(name, "dump_direct")) h->dump_direct = value != 0.0;
    else if (!strcmp(name, "screen")) {
        if (value != 0.0 && value != 1.0 && value != 2.0) return fail(h, MPCB_ERR_INVALID, "screen must be 0, 1 or 2");
        h->screen = (int)value;
    }
    else if (!strcmp(name, "prefilter")) h->prefilter = value != 0.0;
    else if (!strcmp(name, "subtree_cut")) {
        if (value != 0.0 && value != 1.0 && value != 2.0 && value != 3.0) return fail(h, MPCB_ERR_INVALID, "subtree_cut must be 0, 1, 2 or 3");
        h->subtree_cut = (int)value;
    }
    else if (!strcmp(name, "frontier_cap")) {
        if (!(value >= 1.0 && value <= (double)(1ULL << 28))) return fail(h, MPCB_ERR_INVALID, "frontier_cap out of range [1, 2^28]");
        h->frontier_cap = (unsigned long long)value;
    }
    else if (!strcmp(name, "nodes_per_thread")) {
        if (value != 1.0 && value != 2.0 && value != 4.0) return fail(h, MPCB_ERR_INVALID, "nodes_per_thread must be 1, 2 or 4");
        h->npt = (int)value;
    }
    else return fail(h, MPCB_ERR_INVALID, "unknown option '%s'", name);
    return MPCB_OK;
}

int mpcb_set_grid(mpcb_handle *h, const double *v, int nv, const double *beta, int nb, double L, double delta_t,
                  double v_min) {
    if (!h || (!v && nv) || (!beta && nb) || nv < 0 || nb < 0) return fail(h, MPCB_ERR_INVALID, "set_grid: bad arguments");
    if (nv == 0 || nb == 0) { h->have_grid = false; return fail(h, MPCB_ERR_EMPTY_GRID, "empty control grid"); }
    if ((long long)nv * nb > (1LL << 30)) return fail(h, MPCB_ERR_TOO_LARGE, "grid too large");
    // Host-side only: the per-control tables are built and uploaded on first use by a kernel that
    // needs them (ensure_tables); the low-latency HELD path works from the raw grids.
    h->hv.assign(v, v + nv);
    h->hb.assign(beta, beta + nb);
    h->L = L; h->delta_t = delta_t; h->v_min = v_min;
    double vmin_grid = v[0];
    for (int i = 1; i < nv; ++i) vmin_grid = std::min(vmin_grid, v[i]);
    h->v_slow = vmin_grid > v_min ? vmin_grid : v_min;   // math_model_tree.py:312-316
    h->g.S = nv * nb; h->g.nb = nb; h->g.dt = delta_t;
    h->have_grid = true;
    h->tables_ready = false;
    ++h->epoch;
    return MPCB_OK;
}

}  // extern "C"

// The solve behind every batch entry point.  split_comm != null: ONE tree (per solve) shared by the ranks of an NCCL
// communicator -- this rank expands the first controls of its contiguous share, the per-rank (cost, index) records
// are all-gathered (16 bytes per solve and rank, one collective) and every rank finalises the same winner.
static int solve_core(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N, const double *state,
                      const double *target, const double *origin, const double *threshold,
                      const uint8_t *flags, int64_t i0_begin, int64_t i0_end, double *best_cost,
                      int64_t *best_index, double *best_traj, double *first_control, void *split_comm) {
    if (!h) return MPCB_ERR_INVALID;
    if (!h->have_grid) return fail(h, MPCB_ERR_NO_GRID, "mpcb_set_grid has not been called");
    if (H < 1 || H > MPCB_MAX_H) return fail(h, MPCB_ERR_INVALID, "H=%d out of range [1,%d]", H, MPCB_MAX_H);
    if ((mode != MPCB_MODE_FULL && mode != MPCB_MODE_HELD) || (cost_kind != MPCB_COST_MM && cost_kind != MPCB_COST_TREE))
        return fail(h, MPCB_ERR_INVALID, "bad mode/cost");
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (N == 0) return MPCB_OK;
    if (!state || !target || !origin) return fail(h, MPCB_ERR_INVALID, "null input pointer");
    CK(cudaSetDevice(h->device));
    int rc = ensure_tables(h);
    if (rc) return rc;
    int nranks = 1, rank = 0;
    if (split_comm) {
        if (mode != MPCB_MODE_FULL) return fail(h, MPCB_ERR_INVALID, "only a FULL tree is split across ranks");
        if (nccl_comm_info(split_comm, &nranks, &rank) != MPCB_OK) return fail(h, MPCB_ERR_NCCL, "bad NCCL communicator");
        // contiguous, balanced ranges of the first control: rank order = leaf-index order
        const long long S = h->g.S, per = S / nranks, extra = S % nranks;
        i0_begin = rank * per + std::min<long long>(rank, extra);
        i0_end = i0_begin + per + (rank < extra ? 1 : 0);
    }
    Plan pl;
    rc = make_plan(h, mode, H, N, i0_begin, i0_end, MPCB_ALGO_AUTO, pl);
    if (rc) return rc;

    LaunchArgs a;
    fill_args(h, a, mode, cost_kind, H, N, pl);
    const unsigned long long units = pl.u_end - pl.u_begin;
    a.tiles_per_solve = (units + a.tile_units - 1) / a.tile_units;
    fastdiv_init(a.fd_tiles, std::max<unsigned long long>(a.tiles_per_solve, 1));
    fastdiv_init(a.fd_S, (unsigned long long)h->g.S);
    unsigned __int128 all_tiles = (unsigned __int128)a.tiles_per_solve * (unsigned long long)N;
    unsigned long long tps = (unsigned long long)((all_tiles + kSegCap - 1) / kSegCap);
    if (tps < 1) tps = 1;
    if (tps >= (1ULL << 32)) return fail(h, MPCB_ERR_TOO_LARGE, "tree too large for one launch; split by first control");
    a.tps = (unsigned)tps;
    a.segs_per_solve = a.tiles_per_solve ? (a.tiles_per_solve + tps - 1) / tps : 0;
    a.total_segs = a.segs_per_solve * (unsigned long long)N;
    if (a.total_segs >= (1ULL << 32)) return fail(h, MPCB_ERR_TOO_LARGE, "too many segments");

    CK(h->sp.ensure(sizeof(SolveParams) * N));
    CK(h->segmin.ensure(sizeof(double) * std::max<unsigned long long>(a.total_segs, 1)));
    CK(h->worklist.ensure(sizeof(unsigned) * std::max<unsigned long long>(a.total_segs, 1)));
    CK(h->misc.ensure(128));
    CK(h->tau.ensure(sizeof(double) * N));
    CK(h->bestJ.ensure(sizeof(double) * N));
    CK(h->bestIdx.ensure(sizeof(long long) * N));
    CK(h->lock.ensure(sizeof(int) * N));
    CK(h->ub.ensure(sizeof(unsigned long long) * N));
    // misc: [0..3] work_count (u32) | [8..11] tile_count (u32, subtree cut) | [16..47] counters (4 x u64) |
    //       [48..55] frontier counts (2 x u32) | [56..59] frontier overflow flag (u32) | [60..63] candidate count (u32) |
    //       [4..7] listed refinement nodes (u32) | [64..71] next work item of the refinement filter (u64) |
    //       [72..79] nodes that passed stage 1 of the two-stage screen (u64, counters[7])
    unsigned *work_count = h->misc.as<unsigned>();
    unsigned long long *counters = reinterpret_cast<unsigned long long *>(h->misc.as<char>() + 16);
    CK(cudaMemsetAsync(h->misc.p, 0, 128, h->stream));
    // candidate list of the refinement: [cand_cap] candidates + their float64 costs, per-solve key and index (all ones)
    // (the prefix algorithm with a node list evaluates its in-window leaves where the scan finds them -- from the node's
    //  float64 pose, one step each -- which beats listing them and three more launches; measured on cfg2 and cfg4)
    const unsigned cand_cap = (h->cand_auto && pl.prefix && h->node_cap) ? 0u : h->cand_cap;
    if (cand_cap) {
        CK(h->cand.ensure(sizeof(Candidate) * cand_cap));
        CK(h->cand_J.ensure(sizeof(double) * cand_cap));
        CK(h->cand_sel.ensure(2 * sizeof(unsigned long long) * N));
        CK(cudaMemsetAsync(h->cand_sel.p, 0xFF, 2 * sizeof(unsigned long long) * N, h->stream));
    }
    CK(cudaMemsetAsync(h->segmin.p, 0xFF, sizeof(double) * std::max<unsigned long long>(a.total_segs, 1), h->stream));

    a.sp = h->sp.as<SolveParams>();
    a.segmin = h->segmin.as<double>();
    a.worklist = h->worklist.as<unsigned>();
    a.work_count = work_count;
    a.bestJ = h->bestJ.as<double>();
    a.bestIdx = h->bestIdx.as<long long>();
    a.lock = h->lock.as<int>();
    a.counters = counters;
    a.tau = h->tau.as<double>();
    a.ub = h->ub.as<unsigned long long>();
    a.refine_ctr = reinterpret_cast<unsigned long long *>(h->misc.as<char>() + 64);
    if (cand_cap) {
        a.cand = h->cand.as<Candidate>(); a.cand_count = h->misc.as<unsigned>() + 15; a.cand_cap = cand_cap;
        a.cand_J = h->cand_J.as<double>();
        a.cand_key = h->cand_sel.as<unsigned long long>(); a.cand_idx = a.cand_key + N;
    }
    if (pl.prefix && h->node_cap) {
        CK(h->node_list.ensure(sizeof(RefineNode) * (size_t)h->node_cap));
        a.node_list = h->node_list.as<RefineNode>(); a.node_count = h->misc.as<unsigned>() + 1; a.node_cap = h->node_cap;
    }
    a.prune = (pl.prefix && h->prune && H >= 2) ? 1 : 0;
    a.npt = h->npt;
    a.screen = (pl.prefix && !a.prune && H >= 2 && h->npt >= 2) ? h->screen : 0;
    a.prefilter = h->prefilter;

    int launches = 0;
    CK(launch_prep(h->stream, N, state, target, origin, threshold, flags, cost_kind, H, (pl.prefix ? 1 : 0) | (mode == MPCB_MODE_HELD ? 2 : 0),
                   h->g.smax, h->g.dphimax, h->tol_scale, h->sp.as<SolveParams>())); ++launches;
    if (a.prune || a.screen) {   // exact upper bound on every solve's minimum from the S held sequences
        CK(launch_probe(h->stream, a, h->sms)); ++launches;
        if (split_comm) {        // ... of this rank's share: the ranks exchange their bounds (8 bytes per solve and rank)
            CK(h->nccl_scratch.ensure(sizeof(SplitRec) * (size_t)N * (nranks + 1)));
            unsigned long long *all = h->nccl_scratch.as<unsigned long long>();
            if (nccl_allgather_bytes(split_comm, h->ub.p, all, sizeof(unsigned long long) * (size_t)N, h->stream) != MPCB_OK)
                return fail(h, MPCB_ERR_NCCL, "ncclAllGather failed");
            CK(launch_split_ub_min(h->stream, a, all, nranks)); ++launches;
        }
    }
    const unsigned __int128 tiles_all = (unsigned __int128)a.tiles_per_solve * (unsigned long long)N;
    if (a.total_segs > 0 && a.prune && h->subtree_cut && H >= 3 && tiles_all < ((unsigned __int128)1 << 63)) {
        // Subtree cut.  Tile path: batches of tiles go through the depth-(H-2) bound, pass 1 walks the surviving
        // tiles -- all enqueued, no host synchronisation (every grid is persistent over a device-side count).
        // Frontier descent (trees of more than one tile batch, where testing every tile is itself the cost):
        // survivors of depth k expand to depth k+1 down to depth H-2 and pass 1 walks their children; if a frontier
        // outgrew its list, pass 1 returns at once and a fused tile walk (tilewalk_fallback_kernel) takes over --
        // a device-side decision, nothing is read back.
        const unsigned long long all = (unsigned long long)tiles_all;
        const unsigned long long batch = std::min<unsigned long long>(all, kTileBatch);
        unsigned long long deepest = 0;                       // N * S^(H-2): the last frontier if nothing is cut
        const bool ids_fit = pow_checked((unsigned long long)h->g.S, H - 2, deepest) &&
                             (unsigned __int128)deepest * (unsigned long long)N < ((unsigned __int128)1 << 62);
        const bool frontier = ids_fit && (h->subtree_cut == 3 || (h->subtree_cut == 2 && all > kTileBatch));
        const unsigned long long cap = std::min<unsigned long long>(h->frontier_cap, std::max<unsigned long long>(deepest * (unsigned long long)N, 1));
        CK(h->tile_list.ensure(sizeof(unsigned long long) * std::max(batch, frontier ? 2 * cap : 0ULL)));
        unsigned long long *lists = h->tile_list.as<unsigned long long>();
        unsigned *tile_count = h->misc.as<unsigned>() + 2;
        unsigned *q_counts = h->misc.as<unsigned>() + 12;     // two ping-pong counts
        unsigned *q_overflow = h->misc.as<unsigned>() + 14;
        a.q_overflow = q_overflow;
        bool tiles_needed = true;
        if (frontier) {
            a.q_cap = (unsigned)cap;
            a.gate = 1;                                       // pass 1 must not walk a truncated list
            for (int k = 0; k <= H - 3; ++k) {
                unsigned *dst_count = q_counts + (k & 1);
                if (k >= 2) CK(cudaMemsetAsync(dst_count, 0, sizeof(unsigned), h->stream));
                CK(launch_frontier_expand(h->stream, a, k, k ? lists + ((k - 1) & 1) * cap : nullptr, k ? q_counts + ((k - 1) & 1) : nullptr,
                                          lists + (k & 1) * cap, dst_count, q_overflow, h->sms)); ++launches;
            }
            a.q_list = lists + ((H - 3) & 1) * cap;
            a.q_count = q_counts + ((H - 3) & 1);
            CK(launch_pass(h->stream, a, h->row_ab, 1, pl.prefix, h->sms)); ++launches;
            a.q_list = nullptr; a.q_count = nullptr; a.gate = 0;
            // a frontier that outgrew its list: the fused tile walk redoes pass 1 -- decided on the device, the kernel
            // returns at once otherwise; the host never reads the flag
            CK(launch_tilewalk_fallback(h->stream, a, all, h->sms)); ++launches;
            tiles_needed = false;
        }
        if (tiles_needed) {
            a.tile_list = lists;
            a.tile_count = tile_count;
            for (unsigned long long g0 = 0; g0 < all; g0 += batch) {
                if (g0 || frontier) CK(cudaMemsetAsync(tile_count, 0, sizeof(unsigned), h->stream));
                CK(launch_tilecut(h->stream, a, g0, std::min(all, g0 + batch), lists, tile_count, batch)); ++launches;
                CK(launch_pass(h->stream, a, h->row_ab, 1, pl.prefix, h->sms)); ++launches;
            }
            a.tile_list = nullptr; a.tile_count = nullptr;
        }
    } else if (a.total_segs > 0) {
        CK(launch_pass(h->stream, a, h->row_ab, 1, pl.prefix, h->sms)); ++launches;
    }
    if (a.segs_per_solve >= kWideReduceSegs) {   // few solves with many segments each: reduce and compact grid-wide
        CK(h->reduce_scratch.ensure(2 * sizeof(double) * N));
        CK(launch_reduce_compact_wide(h->stream, a, h->tau.as<double>(), h->worklist.as<unsigned>(), work_count,
                                      h->reduce_scratch.p, h->sms, &launches));
    } else {
        CK(launch_reduce_compact(h->stream, a, h->tau.as<double>(), h->worklist.as<unsigned>(), work_count, h->sms)); ++launches;
    }
    if (a.total_segs > 0) {
        CK(launch_pass(h->stream, a, h->row_ab, 2, pl.prefix, h->sms)); ++launches;
        if (a.node_list) { CK(launch_refine_scan(h->stream, a, h->sms)); ++launches; }
        if (a.cand) { CK(launch_cand_resolve(h->stream, a, h->sms)); launches += 3; }
    }
    if (split_comm) {
        CK(h->nccl_scratch.ensure(sizeof(SplitRec) * (size_t)N * (nranks + 1)));
        SplitRec *mine = h->nccl_scratch.as<SplitRec>(), *all = mine + N;
        CK(launch_split_pack(h->stream, a, mine)); ++launches;
        if (nccl_allgather_bytes(split_comm, mine, all, sizeof(SplitRec) * (size_t)N, h->stream) != MPCB_OK)
            return fail(h, MPCB_ERR_NCCL, "ncclAllGather failed");
        CK(launch_split_pick(h->stream, a, all, nranks)); ++launches;
    }
    CK(launch_finalize(h->stream, a, best_cost, (long long *)best_index, best_traj, first_control)); ++launches;

    h->stats.units = (int64_t)units;
    h->stats.leaves_per_solve = (int64_t)pl.leaves_per_solve;
    h->stats.segments = (int64_t)a.total_segs;
    h->stats.algo = pl.prefix ? MPCB_ALGO_PREFIX : MPCB_ALGO_LEAFWALK;
    h->stats.kernel_launches = launches;
    h->stats.refine_segments = -1;   // resolved lazily by mpcb_get_stats
    h->stats.refine_candidates = -1;
    return MPCB_OK;
}

extern "C" {

int mpcb_solve_batch_device(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N, const double *state,
                            const double *target, const double *origin, const double *threshold,
                            const uint8_t *flags, int64_t i0_begin, int64_t i0_end, double *best_cost,
                            int64_t *best_index, double *best_traj, double *first_control) {
    return solve_core(h, mode, cost_kind, H, N, state, target, origin, threshold, flags, i0_begin, i0_end, best_cost,
                      best_index, best_traj, first_control, nullptr);
}

int mpcb_solve_tree_split_device(mpcb_handle *h, void *nccl_comm, int cost_kind, int H, int64_t N, const double *state,
                                 const double *target, const double *origin, const double *threshold,
                                 double *best_cost, int64_t *best_index, double *best_traj, double *first_control) {
    if (!h) return MPCB_ERR_INVALID;
    if (!nccl_comm || !nccl_available()) return fail(h, MPCB_ERR_NCCL, "split tree: no NCCL communicator");
    return solve_core(h, MPCB_MODE_FULL, cost_kind, H, N, state, target, origin, threshold, nullptr, 0, -1, best_cost,
                      best_index, best_traj, first_control, nccl_comm);
}

int mpcb_get_stats(mpcb_handle *h, mpcb_stats *out) {
    if (!h || !out) return MPCB_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (h->stats.refine_segments < 0 && h->misc.p) {
        unsigned long long c[8] = {};
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaMemcpy(c, h->misc.as<char>() + 16, sizeof c, cudaMemcpyDeviceToHost));
        h->stats.refine_segments = (int64_t)c[0];
        h->stats.refine_candidates = (int64_t)c[1];
        h->stats.pruned_units = (int64_t)c[2];
        h->stats.stage2_units = (int64_t)c[7];
    }
    *out = h->stats;
    return MPCB_OK;
}

// Low-latency HELD path of the host API: one pinned staging buffer in, ONE kernel (float64, straight
// from the raw grids), one staging buffer out -- 1 H2D + 1 launch + 1 D2H + 1 sync per call.
static int solve_held_small(mpcb_handle *h, int cost_kind, int H, int64_t N, const double *state,
                            const double *target, const double *origin, const double *threshold,
                            const uint8_t *flags, double *best_cost, int64_t *best_index, double *best_traj,
                            double *first_control) {
    cudaStream_t st = h->stream;
    const size_t nv = h->hv.size(), nb = h->hb.size();
    const size_t n_in = nv + nb + (size_t)N * (3 + 2 + 2 + (threshold ? 1 : 0) + (flags ? 1 : 0));
    const size_t n_out = (size_t)N * (1 + 1 + 3 * H + 2);
    auto pinned = [&](void *&p, size_t &cap, size_t bytes) -> cudaError_t {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaHostAlloc(&p, bytes * 2, cudaHostAllocMapped);
        if (e == cudaSuccess) cap = bytes * 2;
        return e;
    };
    CK(pinned(h->pin_in, h->pin_in_cap, n_in * 8));
    CK(pinned(h->pin_out, h->pin_out_cap, n_out * 8));
    // A tick of a few robots moves a few hundred bytes each way: the kernel reads its inputs from, and writes its
    // results to, MAPPED pinned host memory -- one launch and one synchronisation, no copy engine (option "zero_copy").
    // Bigger batches are staged through device buffers with one copy each way.
    const bool zero_copy = h->zero_copy && N <= 64;
    void *zin = nullptr, *zout = nullptr;
    if (zero_copy) {
        CK(cudaHostGetDevicePointer(&zin, h->pin_in, 0));
        CK(cudaHostGetDevicePointer(&zout, h->pin_out, 0));
    } else {
        CK(h->small_in.ensure(n_in * 8));
        CK(h->small_out.ensure(n_out * 8));
    }
    double *w = (double *)h->pin_in;
    const double *d = zero_copy ? (const double *)zin : h->small_in.as<double>();
    SmallArgs a{};
    auto put = [&](const double *src, size_t cnt) { const double *dev = d + (w - (double *)h->pin_in); memcpy(w, src, cnt * 8); w += cnt; return dev; };
    a.v = put(h->hv.data(), nv);
    a.beta = put(h->hb.data(), nb);
    a.state = put(state, 3 * (size_t)N);
    a.target = put(target, 2 * (size_t)N);
    a.origin = put(origin, 2 * (size_t)N);
    if (threshold) a.threshold = put(threshold, (size_t)N);
    if (flags) {
        a.flags = d + (w - (double *)h->pin_in);
        for (int64_t i = 0; i < N; ++i) *w++ = (double)(flags[i] & (MPCB_FLAG_SLOW | MPCB_FLAG_SKIP));
    }
    double *o = zero_copy ? (double *)zout : h->small_out.as<double>();
    a.out_cost = o; a.out_index = (long long *)(o + N); a.out_traj = o + 2 * N; a.out_ctl = o + 2 * N + 3 * (size_t)H * N;
    a.L = h->L; a.delta_t = h->delta_t; a.v_slow = h->v_slow;
    a.nv = (int)nv; a.nb = (int)nb; a.H = H; a.cost_kind = cost_kind; a.N = N;
    if (!zero_copy) CK(cudaMemcpyAsync(h->small_in.p, h->pin_in, n_in * 8, cudaMemcpyHostToDevice, st));
    CK(launch_held_small(st, a));
    if (!zero_copy) CK(cudaMemcpyAsync(h->pin_out, h->small_out.p, n_out * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const double *r = (const double *)h->pin_out;
    if (best_cost) memcpy(best_cost, r, 8 * (size_t)N);
    if (best_index) memcpy(best_index, r + N, 8 * (size_t)N);
    if (best_traj) memcpy(best_traj, r + 2 * N, 8 * 3 * (size_t)H * N);
    if (first_control) memcpy(first_control, r + 2 * N + 3 * (size_t)H * N, 8 * 2 * (size_t)N);
    h->stats = mpcb_stats{};
    h->stats.units = h->stats.leaves_per_solve = (int64_t)(nv * nb);
    h->stats.algo = MPCB_ALGO_LEAFWALK;
    h->stats.kernel_launches = 1;
    return MPCB_OK;
}

// host buffers -> device staging -> solve_core -> host buffers (one synchronisation)
static int solve_host_staged(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N, const double *state,
                             const double *target, const double *origin, const double *threshold,
                             const uint8_t *flags, int64_t i0_begin, int64_t i0_end, double *best_cost,
                             int64_t *best_index, double *best_traj, double *first_control, void *split_comm) {
    cudaStream_t st = h->stream;
    CK(h->in_state.ensure(sizeof(double) * 3 * N));
    CK(h->in_target.ensure(sizeof(double) * 2 * N));
    CK(h->in_origin.ensure(sizeof(double) * 2 * N));
    CK(cudaMemcpyAsync(h->in_state.p, state, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_target.p, target, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_origin.p, origin, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    const double *d_thr = nullptr;
    const uint8_t *d_flags = nullptr;
    if (threshold) {
        CK(h->in_thr.ensure(sizeof(double) * N));
        CK(cudaMemcpyAsync(h->in_thr.p, threshold, sizeof(double) * N, cudaMemcpyHostToDevice, st));
        d_thr = h->in_thr.as<double>();
    }
    if (flags) {
        CK(h->in_flags.ensure(N));
        CK(cudaMemcpyAsync(h->in_flags.p, flags, N, cudaMemcpyHostToDevice, st));
        d_flags = h->in_flags.as<uint8_t>();
    }
    CK(h->out_cost.ensure(sizeof(double) * N));
    CK(h->out_index.ensure(sizeof(int64_t) * N));
    CK(h->out_traj.ensure(sizeof(double) * 3 * H * N));
    CK(h->out_ctl.ensure(sizeof(double) * 2 * N));
    int rc = solve_core(h, mode, cost_kind, H, N, h->in_state.as<double>(), h->in_target.as<double>(),
                        h->in_origin.as<double>(), d_thr, d_flags, i0_begin, i0_end, h->out_cost.as<double>(),
                        h->out_index.as<int64_t>(), h->out_traj.as<double>(), h->out_ctl.as<double>(), split_comm);
    if (rc) return rc;
    if (best_cost) CK(cudaMemcpyAsync(best_cost, h->out_cost.p, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    if (best_index) CK(cudaMemcpyAsync(best_index, h->out_index.p, sizeof(int64_t) * N, cudaMemcpyDeviceToHost, st));
    if (best_traj) CK(cudaMemcpyAsync(best_traj, h->out_traj.p, sizeof(double) * 3 * H * N, cudaMemcpyDeviceToHost, st));
    if (first_control) CK(cudaMemcpyAsync(first_control, h->out_ctl.p, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return MPCB_OK;
}

static int check_host_args(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N, const double *state,
                           const double *target, const double *origin) {
    if (!state || !target || !origin) return fail(h, MPCB_ERR_INVALID, "null input pointer");
    if (H < 1 || H > MPCB_MAX_H) return fail(h, MPCB_ERR_INVALID, "H=%d out of range [1,%d]", H, MPCB_MAX_H);
    if (!h->have_grid) return fail(h, MPCB_ERR_NO_GRID, "mpcb_set_grid has not been called");
    if ((cost_kind != MPCB_COST_MM && cost_kind != MPCB_COST_TREE) || (mode != MPCB_MODE_FULL && mode != MPCB_MODE_HELD))
        return fail(h, MPCB_ERR_INVALID, "bad mode/cost");
    (void)N;
    return MPCB_OK;
}

int mpcb_solve_batch_host(mpcb_handle *h, int mode, int cost_kind, int H, int64_t N, const double *state,
                          const double *target, const double *origin, const double *threshold,
                          const uint8_t *flags, int64_t i0_begin, int64_t i0_end, double *best_cost,
                          int64_t *best_index, double *best_traj, double *first_control) {
    if (!h) return MPCB_ERR_INVALID;
    if (N <= 0) return N == 0 ? MPCB_OK : fail(h, MPCB_ERR_INVALID, "N < 0");
    int rc = check_host_args(h, mode, cost_kind, H, N, state, target, origin);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if (mode == MPCB_MODE_HELD && h->small_path && h->g.S <= 4096 && h->hb.size() <= 4096 && N <= 8192)
        return solve_held_small(h, cost_kind, H, N, state, target, origin, threshold, flags, best_cost, best_index,
                                best_traj, first_control);
    return solve_host_staged(h, mode, cost_kind, H, N, state, target, origin, threshold, flags, i0_begin, i0_end,
                             best_cost, best_index, best_traj, first_control, nullptr);
}

int mpcb_held_tick_host(mpcb_handle *h, const double *v, int nv, const double *beta, int nb, double L, double delta_t,
                        double v_min, int cost_kind, int H, const double *state, const double *target,
                        const double *origin, double threshold, int flags, double *best_cost, int64_t *best_index,
                        double *best_traj, double *first_control) {
    int rc = mpcb_set_grid(h, v, nv, beta, nb, L, delta_t, v_min);
    if (rc) return rc;
    const uint8_t fl = (uint8_t)flags;
    return mpcb_solve_batch_host(h, MPCB_MODE_HELD, cost_kind, H, 1, state, target, origin, &threshold, &fl, 0, -1,
                                 best_cost, best_index, best_traj, first_control);
}

int mpcb_solve_tree_split_host(mpcb_handle *h, void *nccl_comm, int cost_kind, int H, int64_t N, const double *state,
                               const double *target, const double *origin, const double *threshold,
                               double *best_cost, int64_t *best_index, double *best_traj, double *first_control) {
    if (!h) return MPCB_ERR_INVALID;
    if (!nccl_comm || !nccl_available()) return fail(h, MPCB_ERR_NCCL, "split tree: no NCCL communicator");
    if (N <= 0) return N == 0 ? MPCB_OK : fail(h, MPCB_ERR_INVALID, "N < 0");
    int rc = check_host_args(h, MPCB_MODE_FULL, cost_kind, H, N, state, target, origin);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    return solve_host_staged(h, MPCB_MODE_FULL, cost_kind, H, N, state, target, origin, threshold, nullptr, 0, -1,
                             best_cost, best_index, best_traj, first_control, nccl_comm);
}

int mpcb_dump_leaves_host(mpcb_handle *h, int mode, int cost_kind, int H, int algo, const double *state,
                          const double *target, const double *origin, uint8_t flags, int64_t leaf_begin,
                          int64_t count, float *xy, double *cost) {
    if (!h) return MPCB_ERR_INVALID;
    if (!h->have_grid) return fail(h, MPCB_ERR_NO_GRID, "mpcb_set_grid has not been called");
    if (H < 1 || H > MPCB_MAX_H || count < 0 || leaf_begin < 0 || !state || !target || !origin)
        return fail(h, MPCB_ERR_INVALID, "dump: bad arguments");
    if (count == 0) return MPCB_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    int rc = ensure_tables(h);
    if (rc) return rc;
    Plan pl;
    rc = make_plan(h, mode, H, 1, 0, -1, algo == MPCB_ALGO_AUTO ? MPCB_ALGO_LEAFWALK : algo, pl);
    if (rc) return rc;
    if ((unsigned long long)(leaf_begin + count) > pl.leaves_per_solve)
        return fail(h, MPCB_ERR_INVALID, "dump range exceeds the %llu leaves of the tree", pl.leaves_per_solve);
    LaunchArgs a;
    fill_args(h, a, mode, cost_kind, H, 1, pl);
    CK(h->in_state.ensure(sizeof(double) * 3)); CK(h->in_target.ensure(sizeof(double) * 2));
    CK(h->in_origin.ensure(sizeof(double) * 2)); CK(h->in_flags.ensure(1));
    CK(cudaMemcpyAsync(h->in_state.p, state, sizeof(double) * 3, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_target.p, target, sizeof(double) * 2, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_origin.p, origin, sizeof(double) * 2, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_flags.p, &flags, 1, cudaMemcpyHostToDevice, st));
    CK(h->sp.ensure(sizeof(SolveParams)));
    CK(h->dump_rec.ensure(sizeof(float4) * count));
    CK(h->dump_j.ensure(sizeof(double) * count));
    CK(launch_prep(st, 1, h->in_state.as<double>(), h->in_target.as<double>(), h->in_origin.as<double>(), nullptr,
                   h->in_flags.as<uint8_t>(), cost_kind, H, (pl.prefix ? 1 : 0) | (mode == MPCB_MODE_HELD ? 2 : 0), h->g.smax, h->g.dphimax, h->tol_scale,
                   h->sp.as<SolveParams>()));
    a.sp = h->sp.as<SolveParams>();
    a.dump = h->dump_rec.as<float4>();
    a.dump_begin = (unsigned long long)leaf_begin;
    a.dump_count = (unsigned long long)count;
    // positions always come from the leafwalk kernel; costs from the requested algorithm
    CK(launch_dump(st, a, false, h->dump_j.as<double>(), h->sms));
    std::vector<float4> rec(count);
    std::vector<double> jr(count);
    CK(cudaMemcpyAsync(rec.data(), h->dump_rec.p, sizeof(float4) * count, cudaMemcpyDeviceToHost, st));
    if (pl.prefix) {
        // the prefix flavour needs the prefix-mode SolveParams (tolerance differs only), same anchors
        CK(launch_dump(st, a, true, h->dump_j.as<double>(), h->sms));
    }
    CK(cudaMemcpyAsync(jr.data(), h->dump_j.p, sizeof(double) * count, cudaMemcpyDeviceToHost, st));
    SolveParams P;
    CK(cudaMemcpyAsync(&P, h->sp.p, sizeof P, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < count; ++i) {
        if (xy) { xy[2 * i] = rec[i].x; xy[2 * i + 1] = rec[i].y; }
        if (cost) cost[i] = P.Kbase + jr[i];
    }
    return MPCB_OK;
}

// a closed loop's operator-event script (host memory: it is configuration, like the loop parameters)
static int check_events(mpcb_handle *h, const mpcb_loop_event *events, int32_t n_events) {
    if (n_events < 0 || n_events > 4096 || (n_events > 0 && !events))
        return fail(h, MPCB_ERR_INVALID, "closed loop: bad event script (n_events=%d)", n_events);
    for (int e = 0; e < n_events; ++e)
        if (events[e].kind < MPCB_EVENT_NEW_TARGET || events[e].kind > MPCB_EVENT_TURN_RIGHT)
            return fail(h, MPCB_ERR_INVALID, "closed loop: event %d has unknown kind %d", e, events[e].kind);
    return MPCB_OK;
}

// numpy seeds of N generators: keys[N] integer seeds (key_len 0) or keys[N][key_len] (1 <= key_len <= 4096)
static int check_seed_keys(mpcb_handle *h, int64_t N, const uint32_t *keys, int32_t key_len) {
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (key_len < 0 || key_len > 4096) return fail(h, MPCB_ERR_INVALID, "seeding: key_len %d outside [0, 4096]", key_len);
    if (N > 0 && !keys) return fail(h, MPCB_ERR_INVALID, "seeding: null keys");
    return MPCB_OK;
}

// numpy SeedSequence words of N PCG64 generators: entropy[entropy_len] shared (stride 0) or [N][entropy_len], and
// spawn_key[N][spawn_len] (spawn_len 0: none); 1 <= entropy_len <= 4096, 0 <= spawn_len <= 4096
static int check_pcg64_seeds(mpcb_handle *h, int64_t N, const uint32_t *entropy, int32_t entropy_len,
                             int32_t entropy_stride, const uint32_t *spawn_key, int32_t spawn_len) {
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (entropy_len < 1 || entropy_len > 4096)
        return fail(h, MPCB_ERR_INVALID, "PCG64 seeding: entropy_len %d outside [1, 4096]", entropy_len);
    if (entropy_stride != 0 && entropy_stride != entropy_len)
        return fail(h, MPCB_ERR_INVALID, "PCG64 seeding: entropy_stride %d is neither 0 nor entropy_len", entropy_stride);
    if (spawn_len < 0 || spawn_len > 4096)
        return fail(h, MPCB_ERR_INVALID, "PCG64 seeding: spawn_len %d outside [0, 4096]", spawn_len);
    if (N > 0 && (!entropy || (spawn_len > 0 && !spawn_key)))
        return fail(h, MPCB_ERR_INVALID, "PCG64 seeding: null seed words");
    return MPCB_OK;
}

// a PCG64 record as numpy could hold it: has_uint32 0/1, uinteger of 32 bits, inc odd
static int check_pcg64_states(mpcb_handle *h, int64_t N, const uint64_t *pcg_state) {
    for (int64_t n = 0; n < N; ++n) {
        const uint64_t *r = pcg_state + n * mpcb::kPcgWords;
        if (r[4] > 1 || r[5] > 0xffffffffull || !(r[3] & 1))
            return fail(h, MPCB_ERR_INVALID, "PCG64 closed loop: robot %lld has a record numpy cannot hold (has_uint32 %llu, "
                        "uinteger %llu, inc %s)", (long long)n, (unsigned long long)r[4], (unsigned long long)r[5],
                        (r[3] & 1) ? "odd" : "even");
    }
    return MPCB_OK;
}

// the trace of this closed-loop call, detached from the handle: one call consumes it, whatever its outcome
static mpcb_loop_trace take_trace(mpcb_handle *h) {
    const mpcb_loop_trace t = h->trace;
    h->trace = mpcb_loop_trace{};
    return t;
}

int mpcb_set_loop_trace(mpcb_handle *h, const mpcb_loop_trace *trace) {
    if (!h) return MPCB_ERR_INVALID;
    h->trace = trace ? *trace : mpcb_loop_trace{};
    return MPCB_OK;
}

// the ranges of a closed loop's parameters
static int check_loop_params(mpcb_handle *h, const mpcb_loop_params *p) {
    if (p->H < 1 || p->H > MPCB_MAX_H || p->max_ticks < 1 || p->n_v < 1 || p->n_beta < 1 || p->n_v > 128 || p->n_beta > 128)
        return fail(h, MPCB_ERR_INVALID, "closed loop: bad parameters (H=%d, max_ticks=%d, n_v=%d, n_beta=%d)", p->H,
                    p->max_ticks, p->n_v, p->n_beta);
    return MPCB_OK;
}

// device pointers throughout, except the event script (checked by the caller with check_events), which is copied into
// handle scratch here; events / out_final / rng_state / pcg_state and the trace's members may be null (at most one of
// rng_state and pcg_state is not)
static int held_loop_core(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                          const double *target, const double *origin, const double *first_threshold,
                          const int32_t *slow_steps, const mpcb_loop_event *events, int n_events, double radius_u_turn,
                          uint32_t *rng_state, double *out_log, int32_t *out_ticks, int32_t *out_status,
                          double *out_final, uint64_t *pcg_state, const mpcb_loop_trace &tr) {
    if (!h || !p) return MPCB_ERR_INVALID;
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (N == 0) return MPCB_OK;
    if (!init || !target || !origin || !out_log || !out_ticks || !out_status)
        return fail(h, MPCB_ERR_INVALID, "closed loop: null pointer");
    int rc = check_loop_params(h, p);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const mpcb_loop_event *d_events = nullptr;
    if (events && n_events > 0) {
        CK(h->loop_events.ensure(sizeof(mpcb_loop_event) * n_events));
        CK(cudaMemcpyAsync(h->loop_events.p, events, sizeof(mpcb_loop_event) * n_events, cudaMemcpyHostToDevice, h->stream));
        d_events = h->loop_events.as<mpcb_loop_event>();
    }
    LoopArgs a;
    a.p = *p; a.N = N;
    a.init = init; a.target = target; a.origin = origin; a.first_threshold = first_threshold;
    a.slow_steps = slow_steps; a.out_log = out_log; a.out_ticks = out_ticks; a.out_status = out_status;
    a.events = d_events; a.n_events = d_events ? n_events : 0; a.radius_u_turn = radius_u_turn; a.out_final = out_final;
    a.rng_state = rng_state;
    a.pcg_state = reinterpret_cast<unsigned long long *>(pcg_state);
    a.trace_pred = tr.pred; a.trace_ctl = tr.control; a.trace_cost = tr.cost;
    CK(launch_held_loop(h->stream, a, h->sms));
    h->stats = mpcb_stats{};
    h->stats.kernel_launches = 1;
    h->stats.algo = MPCB_ALGO_LEAFWALK;
    return MPCB_OK;
}

int mpcb_held_closed_loop_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                 const double *target, const double *origin, const double *first_threshold,
                                 const int32_t *slow_steps, double *out_log, int32_t *out_ticks, int32_t *out_status) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    return held_loop_core(h, p, N, init, target, origin, first_threshold, slow_steps, nullptr, 0, 0.0, nullptr, out_log,
                          out_ticks, out_status, nullptr, nullptr, tr);
}

int mpcb_held_closed_loop_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                               const double *target, const double *origin, const double *first_threshold,
                               const int32_t *slow_steps, double *out_log, int32_t *out_ticks, int32_t *out_status) {
    return mpcb_held_closed_loop_events_host(h, p, N, init, target, origin, first_threshold, slow_steps, nullptr, 0, 0.0,
                                             out_log, out_ticks, out_status, nullptr);
}

// the host trace tr of nrow = N * max_ticks rows in handle scratch, NaN-filled (dtr: its device twin, members null
// where tr's are)
static int stage_trace(mpcb_handle *h, const mpcb_loop_trace &tr, size_t nrow, int H, mpcb_loop_trace &dtr) {
    dtr = mpcb_loop_trace{};
    if (!tr.pred && !tr.control && !tr.cost) return MPCB_OK;
    if (H < 1 || H > MPCB_MAX_H) return fail(h, MPCB_ERR_INVALID, "closed loop trace: H=%d out of range", H);
    cudaStream_t st = h->stream;
    auto one = [&](double *host, mpcb::DevBuf &buf, size_t n, double *&dev) -> cudaError_t {
        if (!host) return cudaSuccess;
        cudaError_t e = buf.ensure(sizeof(double) * n);
        if (e == cudaSuccess) e = cudaMemsetAsync(buf.p, 0xFF, sizeof(double) * n, st);
        dev = buf.as<double>();
        return e;
    };
    CK(one(tr.pred, h->trace_pred, nrow * 3 * H, dtr.pred));
    CK(one(tr.control, h->trace_ctl, nrow * 2, dtr.control));
    CK(one(tr.cost, h->trace_cost, nrow, dtr.cost));
    return MPCB_OK;
}

static cudaError_t copy_back_trace(mpcb_handle *h, const mpcb_loop_trace &tr, const mpcb_loop_trace &dtr, size_t nrow,
                                   int H) {
    cudaError_t e = cudaSuccess;
    if (tr.pred) e = cudaMemcpyAsync(tr.pred, dtr.pred, sizeof(double) * nrow * 3 * H, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && tr.control)
        e = cudaMemcpyAsync(tr.control, dtr.control, sizeof(double) * nrow * 2, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && tr.cost)
        e = cudaMemcpyAsync(tr.cost, dtr.cost, sizeof(double) * nrow, cudaMemcpyDeviceToHost, h->stream);
    return e;
}

// the PCG64 generators of held_loop_host: copied in from state_in[N][6] or seeded on the device from SeedSequence
// words (entropy != null, as for mpcb_pcg64_seed_device); state_out[N][6] (nullable) receives them after the run
struct PcgSource {
    const uint64_t *state_in = nullptr;
    const uint32_t *entropy = nullptr, *spawn_key = nullptr;
    int32_t entropy_len = 0, entropy_stride = 0, spawn_len = 0;
    uint64_t *state_out = nullptr;
    bool any() const { return state_in || entropy; }
};

// host pointers.  The actual run's generators are copied in from rng_in[N][625] or seeded on the device from keys
// (key_len as for mpcb_rng_seed_device), or are PCG64 ones (pcg); with none of them, the loop is the noise-free one.
// rng_out[N][625] (nullable) receives the MT19937 generators' states after the run; the trace (host pointers) is staged
// on the device, NaN-filled as the log is, and copied back.
static int held_loop_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init, const double *target,
                          const double *origin, const double *first_threshold, const int32_t *slow_steps,
                          const mpcb_loop_event *events, int32_t n_events, double radius_u_turn, const uint32_t *rng_in,
                          const uint32_t *keys, int32_t key_len, uint32_t *rng_out, double *out_log, int32_t *out_ticks,
                          int32_t *out_status, double *out_final, const mpcb_loop_trace &tr,
                          const PcgSource &pcg = PcgSource()) {
    int rc = check_events(h, events, n_events);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? MPCB_OK : fail(h, MPCB_ERR_INVALID, "N < 0");
    if (!init || !target || !origin || !out_log || !out_ticks || !out_status)
        return fail(h, MPCB_ERR_INVALID, "closed loop: null pointer");
    if (p->max_ticks < 1) return fail(h, MPCB_ERR_INVALID, "closed loop: max_ticks < 1");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const size_t nlog = (size_t)N * p->max_ticks * 5;
    CK(h->in_state.ensure(sizeof(double) * 5 * N));
    CK(h->in_target.ensure(sizeof(double) * 2 * N));
    CK(h->in_origin.ensure(sizeof(double) * 2 * N));
    CK(h->loop_log.ensure(sizeof(double) * nlog));
    CK(h->loop_ticks.ensure(sizeof(int) * N));
    CK(h->loop_status.ensure(sizeof(int) * N));
    CK(cudaMemcpyAsync(h->in_state.p, init, sizeof(double) * 5 * N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_target.p, target, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_origin.p, origin, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    const double *d_thr = nullptr;
    const int *d_slow = nullptr;
    if (first_threshold) {
        CK(h->in_thr.ensure(sizeof(double) * N));
        CK(cudaMemcpyAsync(h->in_thr.p, first_threshold, sizeof(double) * N, cudaMemcpyHostToDevice, st));
        d_thr = h->in_thr.as<double>();
    }
    if (slow_steps) {
        CK(h->in_flags.ensure(sizeof(int) * N));
        CK(cudaMemcpyAsync(h->in_flags.p, slow_steps, sizeof(int) * N, cudaMemcpyHostToDevice, st));
        d_slow = h->in_flags.as<int>();
    }
    const size_t nrng = (size_t)N * mpcb::kMtWords;
    const bool noise = rng_in || keys;
    if (noise) CK(h->loop_rng.ensure(sizeof(uint32_t) * nrng));
    if (rng_in) CK(cudaMemcpyAsync(h->loop_rng.p, rng_in, sizeof(uint32_t) * nrng, cudaMemcpyHostToDevice, st));
    if (keys) {
        const size_t nkeys = (size_t)N * (key_len ? key_len : 1);
        CK(h->loop_keys.ensure(sizeof(uint32_t) * nkeys));
        CK(cudaMemcpyAsync(h->loop_keys.p, keys, sizeof(uint32_t) * nkeys, cudaMemcpyHostToDevice, st));
        CK(launch_rng_seed(st, N, h->loop_keys.as<unsigned>(), key_len, h->loop_rng.as<unsigned>()));
    }
    const size_t npcg = (size_t)N * mpcb::kPcgWords;
    if (pcg.any()) CK(h->loop_pcg.ensure(sizeof(uint64_t) * npcg));
    if (pcg.state_in)
        CK(cudaMemcpyAsync(h->loop_pcg.p, pcg.state_in, sizeof(uint64_t) * npcg, cudaMemcpyHostToDevice, st));
    if (pcg.entropy) {      // the entropy words go to loop_keys, the spawn-key words to loop_pcg_spawn
        const size_t nent = (size_t)(pcg.entropy_stride ? N : 1) * pcg.entropy_len;
        CK(h->loop_keys.ensure(sizeof(uint32_t) * nent));
        CK(cudaMemcpyAsync(h->loop_keys.p, pcg.entropy, sizeof(uint32_t) * nent, cudaMemcpyHostToDevice, st));
        const unsigned *d_spawn = nullptr;
        if (pcg.spawn_len > 0) {
            const size_t nsp = (size_t)N * pcg.spawn_len;
            CK(h->loop_pcg_spawn.ensure(sizeof(uint32_t) * nsp));
            CK(cudaMemcpyAsync(h->loop_pcg_spawn.p, pcg.spawn_key, sizeof(uint32_t) * nsp, cudaMemcpyHostToDevice, st));
            d_spawn = h->loop_pcg_spawn.as<unsigned>();
        }
        CK(launch_pcg64_seed(st, N, h->loop_keys.as<unsigned>(), pcg.entropy_len, pcg.entropy_stride, d_spawn,
                             pcg.spawn_len, h->loop_pcg.as<unsigned long long>()));
    }
    if (out_final) CK(h->loop_final.ensure(sizeof(double) * 6 * N));
    CK(cudaMemsetAsync(h->loop_log.p, 0xFF, sizeof(double) * nlog, st));     // NaN pattern for the rows no tick wrote
    const size_t nrow = (size_t)N * p->max_ticks;
    mpcb_loop_trace dtr{};
    rc = stage_trace(h, tr, nrow, p->H, dtr);
    if (rc) return rc;
    rc = held_loop_core(h, p, N, h->in_state.as<double>(), h->in_target.as<double>(), h->in_origin.as<double>(), d_thr,
                        d_slow, events, n_events, radius_u_turn, noise ? h->loop_rng.as<uint32_t>() : nullptr,
                        h->loop_log.as<double>(), h->loop_ticks.as<int>(), h->loop_status.as<int>(),
                        out_final ? h->loop_final.as<double>() : nullptr, pcg.any() ? h->loop_pcg.as<uint64_t>() : nullptr,
                        dtr);
    if (rc) return rc;
    if (keys || pcg.entropy) h->stats.kernel_launches += 1;     // the seeding kernel
    if (rng_out) CK(cudaMemcpyAsync(rng_out, h->loop_rng.p, sizeof(uint32_t) * nrng, cudaMemcpyDeviceToHost, st));
    if (pcg.state_out)
        CK(cudaMemcpyAsync(pcg.state_out, h->loop_pcg.p, sizeof(uint64_t) * npcg, cudaMemcpyDeviceToHost, st));
    if (out_final) CK(cudaMemcpyAsync(out_final, h->loop_final.p, sizeof(double) * 6 * N, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_log, h->loop_log.p, sizeof(double) * nlog, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_ticks, h->loop_ticks.p, sizeof(int) * N, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_status, h->loop_status.p, sizeof(int) * N, cudaMemcpyDeviceToHost, st));
    CK(copy_back_trace(h, tr, dtr, nrow, p->H));
    CK(cudaStreamSynchronize(st));
    return MPCB_OK;
}

int mpcb_held_closed_loop_events_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                      const double *target, const double *origin, const double *first_threshold,
                                      const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                      double radius_u_turn, double *out_log, int32_t *out_ticks, int32_t *out_status,
                                      double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    return held_loop_host(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          nullptr, nullptr, 0, nullptr, out_log, out_ticks, out_status, out_final, tr);
}

int mpcb_held_closed_loop_actual_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                      const double *target, const double *origin, const double *first_threshold,
                                      const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                      double radius_u_turn, uint32_t *rng_state, double *out_log, int32_t *out_ticks,
                                      int32_t *out_status, double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    if (!rng_state) return fail(h, MPCB_ERR_INVALID, "actual closed loop: null rng_state");
    for (int64_t n = 0; n < N; ++n) {
        const uint32_t pos = rng_state[n * mpcb::kMtWords + mpcb::kMtN];
        if (pos > (uint32_t)mpcb::kMtN)
            return fail(h, MPCB_ERR_INVALID, "actual closed loop: robot %lld has generator position %u (outside [0, 624])",
                        (long long)n, pos);
    }
    return held_loop_host(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          rng_state, nullptr, 0, rng_state, out_log, out_ticks, out_status, out_final, tr);
}

int mpcb_held_closed_loop_actual_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                        const double *target, const double *origin, const double *first_threshold,
                                        const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                        double radius_u_turn, uint32_t *rng_state, double *out_log, int32_t *out_ticks,
                                        int32_t *out_status, double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    int rc = check_events(h, events, n_events);
    if (rc) return rc;
    if (!rng_state) return fail(h, MPCB_ERR_INVALID, "actual closed loop: null rng_state");
    return held_loop_core(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          rng_state, out_log, out_ticks, out_status, out_final, nullptr, tr);
}

int mpcb_held_closed_loop_seeded_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                      const double *target, const double *origin, const double *first_threshold,
                                      const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                      double radius_u_turn, const uint32_t *keys, int32_t key_len,
                                      uint32_t *rng_state_out, double *out_log, int32_t *out_ticks, int32_t *out_status,
                                      double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    int rc = check_seed_keys(h, N, keys, key_len);
    if (rc) return rc;
    return held_loop_host(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          nullptr, keys, key_len, rng_state_out, out_log, out_ticks, out_status, out_final, tr);
}

int mpcb_rng_seed_device(mpcb_handle *h, int64_t N, const uint32_t *keys, int32_t key_len, uint32_t *rng_state) {
    if (!h) return MPCB_ERR_INVALID;
    int rc = check_seed_keys(h, N, keys, key_len);
    if (rc) return rc;
    if (N == 0) return MPCB_OK;
    if (!rng_state) return fail(h, MPCB_ERR_INVALID, "seeding: null rng_state");
    CK(cudaSetDevice(h->device));
    CK(launch_rng_seed(h->stream, N, keys, key_len, rng_state));
    return MPCB_OK;
}

int mpcb_held_closed_loop_pcg64_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                     const double *target, const double *origin, const double *first_threshold,
                                     const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                     double radius_u_turn, uint64_t *pcg_state, double *out_log, int32_t *out_ticks,
                                     int32_t *out_status, double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    if (!pcg_state) return fail(h, MPCB_ERR_INVALID, "PCG64 closed loop: null pcg_state");
    int rc = check_pcg64_states(h, N, pcg_state);
    if (rc) return rc;
    PcgSource pcg;
    pcg.state_in = pcg_state;
    pcg.state_out = pcg_state;
    return held_loop_host(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          nullptr, nullptr, 0, nullptr, out_log, out_ticks, out_status, out_final, tr, pcg);
}

int mpcb_held_closed_loop_pcg64_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                       const double *target, const double *origin, const double *first_threshold,
                                       const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                       double radius_u_turn, uint64_t *pcg_state, double *out_log, int32_t *out_ticks,
                                       int32_t *out_status, double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    int rc = check_events(h, events, n_events);
    if (rc) return rc;
    if (!pcg_state) return fail(h, MPCB_ERR_INVALID, "PCG64 closed loop: null pcg_state");
    return held_loop_core(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          nullptr, out_log, out_ticks, out_status, out_final, pcg_state, tr);
}

int mpcb_held_closed_loop_pcg64_seeded_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                                            const double *target, const double *origin, const double *first_threshold,
                                            const int32_t *slow_steps, const mpcb_loop_event *events, int32_t n_events,
                                            double radius_u_turn, const uint32_t *entropy, int32_t entropy_len,
                                            int32_t entropy_stride, const uint32_t *spawn_key, int32_t spawn_len,
                                            uint64_t *pcg_state_out, double *out_log, int32_t *out_ticks,
                                            int32_t *out_status, double *out_final) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (!p) return MPCB_ERR_INVALID;
    int rc = check_pcg64_seeds(h, N, entropy, entropy_len, entropy_stride, spawn_key, spawn_len);
    if (rc) return rc;
    PcgSource pcg;
    pcg.entropy = entropy; pcg.entropy_len = entropy_len; pcg.entropy_stride = entropy_stride;
    pcg.spawn_key = spawn_len > 0 ? spawn_key : nullptr; pcg.spawn_len = spawn_len;
    pcg.state_out = pcg_state_out;
    return held_loop_host(h, p, N, init, target, origin, first_threshold, slow_steps, events, n_events, radius_u_turn,
                          nullptr, nullptr, 0, nullptr, out_log, out_ticks, out_status, out_final, tr, pcg);
}

int mpcb_pcg64_seed_device(mpcb_handle *h, int64_t N, const uint32_t *entropy, int32_t entropy_len,
                           int32_t entropy_stride, const uint32_t *spawn_key, int32_t spawn_len, uint64_t *pcg_state) {
    if (!h) return MPCB_ERR_INVALID;
    int rc = check_pcg64_seeds(h, N, entropy, entropy_len, entropy_stride, spawn_key, spawn_len);
    if (rc) return rc;
    if (N == 0) return MPCB_OK;
    if (!pcg_state) return fail(h, MPCB_ERR_INVALID, "PCG64 seeding: null pcg_state");
    CK(cudaSetDevice(h->device));
    CK(launch_pcg64_seed(h->stream, N, entropy, entropy_len, entropy_stride, spawn_len > 0 ? spawn_key : nullptr,
                         spawn_len, reinterpret_cast<unsigned long long *>(pcg_state)));
    return MPCB_OK;
}

int mpcb_held_ctrl_init_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *init,
                               const double *target, const double *origin, const double *first_threshold,
                               const int32_t *slow_steps, mpcb_held_ctrl *ctrl) {
    if (!h || !p) return MPCB_ERR_INVALID;
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (N == 0) return MPCB_OK;
    if (!init || !target || !origin || !ctrl) return fail(h, MPCB_ERR_INVALID, "controller records: null pointer");
    int rc = check_loop_params(h, p);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    CK(launch_held_ctrl_init(h->stream, N, init, target, origin, first_threshold, slow_steps, ctrl));
    h->stats = mpcb_stats{};
    h->stats.kernel_launches = 1;
    return MPCB_OK;
}

int mpcb_held_ctrl_step_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, mpcb_held_ctrl *ctrl,
                               const double *measured, const mpcb_loop_event *events, int32_t n_ev,
                               double radius_u_turn, double *proposal, int32_t *running) {
    if (!h || !p) return MPCB_ERR_INVALID;
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (n_ev < 0 || n_ev > 64 || (n_ev > 0 && !events))
        return fail(h, MPCB_ERR_INVALID, "controller step: bad events (n_ev=%d, events %s)", n_ev, events ? "set" : "null");
    if (N == 0) return MPCB_OK;
    if (!ctrl) return fail(h, MPCB_ERR_INVALID, "controller step: null records");
    int rc = check_loop_params(h, p);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    HeldCtrlArgs a{};
    a.p = *p; a.N = N; a.ctrl = ctrl; a.measured = measured;
    a.events = n_ev > 0 ? events : nullptr; a.n_ev = n_ev > 0 ? n_ev : 0; a.radius_u_turn = radius_u_turn;
    a.proposal = proposal; a.running = running;
    CK(launch_held_ctrl_step(h->stream, a, h->sms));
    h->stats = mpcb_stats{};
    h->stats.kernel_launches = 1;
    h->stats.algo = MPCB_ALGO_LEAFWALK;
    return MPCB_OK;
}

static int check_window_params(mpcb_handle *h, const mpcb_loop_params *p) {
    if (p->H < 1 || p->H > MPCB_MAX_H || p->n_v < 1 || p->n_beta < 1 || p->n_v > 128 || p->n_beta > 128 ||
        (p->cost_kind != MPCB_COST_MM && p->cost_kind != MPCB_COST_TREE))
        return fail(h, MPCB_ERR_INVALID, "window parameters out of range (H=%d, n_v=%d, n_beta=%d, cost=%d)", p->H, p->n_v,
                    p->n_beta, p->cost_kind);
    return MPCB_OK;
}

int mpcb_solve_held_windows_device(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *state,
                                   const double *v_beta, const double *target, const double *origin,
                                   const double *threshold, const uint8_t *flags, double *best_cost,
                                   int64_t *best_index, double *best_traj, double *first_control, int32_t *window_shape) {
    if (!h || !p) return MPCB_ERR_INVALID;
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (N == 0) return MPCB_OK;
    if (!state || !v_beta || !target || !origin) return fail(h, MPCB_ERR_INVALID, "null input pointer");
    int rc = check_window_params(h, p);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    WindowArgs a{};
    a.p = *p; a.N = N;
    a.state = state; a.vbeta = v_beta; a.target = target; a.origin = origin; a.threshold = threshold; a.flags = flags;
    a.out_cost = best_cost; a.out_index = (long long *)best_index; a.out_traj = best_traj; a.out_ctl = first_control;
    a.out_shape = window_shape;
    CK(launch_held_windows(h->stream, a, h->sms));
    h->stats = mpcb_stats{};
    h->stats.kernel_launches = 1;
    h->stats.algo = MPCB_ALGO_LEAFWALK;
    h->stats.units = h->stats.leaves_per_solve = (int64_t)p->n_v * p->n_beta;
    return MPCB_OK;
}

int mpcb_solve_held_windows_host(mpcb_handle *h, const mpcb_loop_params *p, int64_t N, const double *state,
                                 const double *v_beta, const double *target, const double *origin,
                                 const double *threshold, const uint8_t *flags, double *best_cost,
                                 int64_t *best_index, double *best_traj, double *first_control, int32_t *window_shape) {
    if (!h || !p) return MPCB_ERR_INVALID;
    if (N <= 0) return N == 0 ? MPCB_OK : fail(h, MPCB_ERR_INVALID, "N < 0");
    if (!state || !v_beta || !target || !origin) return fail(h, MPCB_ERR_INVALID, "null input pointer");
    int rc = check_window_params(h, p);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    // one staging buffer each way: [state 3 | v_beta 2 | target 2 | origin 2 | threshold 1] doubles + flags
    const size_t per_in = 3 + 2 + 2 + 2 + (threshold ? 1 : 0);
    const int Hh = p->H;
    const size_t per_out = 1 + 1 + 3 * (size_t)Hh + 2 + 1;       // cost, index, traj, control, shape (2 x int32)
    CK(h->small_in.ensure(sizeof(double) * per_in * N + (flags ? N : 0)));
    CK(h->small_out.ensure(sizeof(double) * per_out * N));
    double *din = h->small_in.as<double>();
    size_t off = 0;
    auto up = [&](const double *src, size_t per) -> const double * {
        const double *dst = din + off;
        cudaMemcpyAsync(din + off, src, sizeof(double) * per * N, cudaMemcpyHostToDevice, st);
        off += per * N;
        return dst;
    };
    const double *d_state = up(state, 3), *d_vb = up(v_beta, 2), *d_target = up(target, 2), *d_origin = up(origin, 2);
    const double *d_thr = threshold ? up(threshold, 1) : nullptr;
    const uint8_t *d_flags = nullptr;
    if (flags) {
        d_flags = reinterpret_cast<const uint8_t *>(din + off);
        cudaMemcpyAsync(din + off, flags, N, cudaMemcpyHostToDevice, st);
    }
    CK(cudaGetLastError());
    double *o = h->small_out.as<double>();
    double *d_cost = o, *d_traj = o + 2 * N, *d_ctl = d_traj + 3 * (size_t)Hh * N;
    int64_t *d_index = reinterpret_cast<int64_t *>(o + N);
    int32_t *d_shape = reinterpret_cast<int32_t *>(d_ctl + 2 * N);
    rc = mpcb_solve_held_windows_device(h, p, N, d_state, d_vb, d_target, d_origin, d_thr, d_flags, d_cost, d_index,
                                        d_traj, d_ctl, d_shape);
    if (rc) return rc;
    if (best_cost) CK(cudaMemcpyAsync(best_cost, d_cost, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    if (best_index) CK(cudaMemcpyAsync(best_index, d_index, sizeof(int64_t) * N, cudaMemcpyDeviceToHost, st));
    if (best_traj) CK(cudaMemcpyAsync(best_traj, d_traj, sizeof(double) * 3 * Hh * N, cudaMemcpyDeviceToHost, st));
    if (first_control) CK(cudaMemcpyAsync(first_control, d_ctl, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, st));
    if (window_shape) CK(cudaMemcpyAsync(window_shape, d_shape, sizeof(int32_t) * 2 * N, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return MPCB_OK;
}

// Destroys the replaced FULL loop graphs, when the handle's stream is idle (all: the caller has just synchronised it).
// cudaGraphExecDestroy waits for the work in flight, which the device entry must not.
static void retire_loop_graphs(mpcb_handle *h, bool all) {
    if (h->fl_graphs.empty()) return;
    if (!all) {
        const cudaError_t q = cudaStreamQuery(h->stream);
        if (q == cudaErrorNotReady && cudaPeekAtLastError() == cudaErrorNotReady)
            (void)cudaGetLastError();            // the query's own "not ready", not an error of a launch
        if (q != cudaSuccess) return;
    }
    for (cudaGraphExec_t x : h->fl_graphs) cudaGraphExecDestroy(x);
    h->fl_graphs.clear();
}

// Launches the handle's FULL loop graph, after destroying replaced ones while the stream is still idle.
static int launch_loop_graph(mpcb_handle *h) {
    retire_loop_graphs(h, false);
    const cudaError_t e = cudaGraphLaunch(h->fl_exec, h->stream);
    if (e != cudaSuccess) return fail(h, MPCB_ERR_CUDA, "full closed loop: graph launch failed: %s", cudaGetErrorString(e));
    return MPCB_OK;
}

// Capture of the FULL loop into g (empty on entry):
//   [running = tick = 0] -> [init] -> [gate] -> WHILE (running > 0 && tick < max_ticks) {
//       solve_core (as it is, every launch and memset of one batched solve) -> [apply] -> [gate] }
// (the gate zeroes the running count after reading it)
// Every capture begun here is ended here, also on failure.  *per_tick: the kernels one tick launches.
static int capture_full_loop(mpcb_handle *h, cudaGraph_t g, const FullLoopArgs &fa, int cost_kind, const double *init,
                             const double *origin, const double *first_threshold, int *per_tick) {
    cudaStream_t st = h->stream;
    int *ctl = fa.active_count;          // [0] running robots, [1] tick
    cudaGraphConditionalHandle cond;
    CK(cudaGraphConditionalHandleCreate(&cond, g, 0, 0));
    CK(cudaStreamBeginCaptureToGraph(st, g, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
    cudaError_t e = cudaMemsetAsync(ctl, 0, 2 * sizeof(int), st);
    if (e == cudaSuccess) e = launch_full_loop_init(st, fa, init, first_threshold);
    if (e == cudaSuccess) e = launch_full_loop_gate(st, cond, ctl, fa.max_ticks, 0);
    cudaGraph_t body = nullptr;
    if (e == cudaSuccess) {              // the WHILE node after the gate
        cudaStreamCaptureStatus cs;
        const cudaGraphNode_t *deps = nullptr;
        size_t ndeps = 0;
        e = cudaStreamGetCaptureInfo(st, &cs, nullptr, nullptr, &deps, &ndeps);
        cudaGraphNodeParams cp = {};
        cp.type = cudaGraphNodeTypeConditional;
        cp.conditional.handle = cond;
        cp.conditional.type = cudaGraphCondTypeWhile;
        cp.conditional.size = 1;
        cudaGraphNode_t node;
        if (e == cudaSuccess) e = cudaGraphAddNode(&node, g, deps, ndeps, &cp);
        if (e == cudaSuccess) e = cudaStreamUpdateCaptureDependencies(st, &node, 1, cudaStreamSetCaptureDependencies);
        if (e == cudaSuccess) body = cp.conditional.phGraph_out[0];
    }
    cudaGraph_t captured = nullptr;
    const cudaError_t e_end = cudaStreamEndCapture(st, &captured);
    if (e != cudaSuccess || e_end != cudaSuccess)
        return fail(h, MPCB_ERR_CUDA, "full closed loop: building the loop graph failed: %s",
                    cudaGetErrorString(e != cudaSuccess ? e : e_end));

    CK(cudaStreamBeginCaptureToGraph(st, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
    int rc = solve_core(h, MPCB_MODE_FULL, cost_kind, fa.H, fa.N, fa.state, fa.target, origin, fa.threshold, fa.flags, 0,
                        -1, h->out_cost.as<double>(), h->out_index.as<int64_t>(), h->out_traj.as<double>(),
                        h->out_ctl.as<double>(), nullptr);
    if (e == cudaSuccess && rc == MPCB_OK) {
        *per_tick = h->stats.kernel_launches + 1;
        e = launch_full_apply(st, fa);
    }
    if (e == cudaSuccess && rc == MPCB_OK) e = launch_full_loop_gate(st, cond, ctl, fa.max_ticks, 1);
    const cudaError_t e_body = cudaStreamEndCapture(st, &captured);
    if (rc) return rc;
    if (e != cudaSuccess || e_body != cudaSuccess)
        return fail(h, MPCB_ERR_CUDA, "full closed loop: capturing the tick failed: %s",
                    cudaGetErrorString(e != cudaSuccess ? e : e_body));
    return MPCB_OK;
}

// The FULL closed loop as ONE graph launch on the handle's stream; device pointers throughout, nothing synchronised.
// N >= 1 and the pointers are checked by the caller; first_threshold and the trace's members are nullable.  The
// executable graph is kept in the handle and launched again while nothing it froze at capture has changed (the key:
// grid and options through the handle's epoch, the handle's buffers through the allocation count, the arguments);
// otherwise the loop is captured and instantiated anew and the old graph destroyed once its last run has ended.
// *per_tick: the kernels one tick launches (the solve's and the apply kernel).
static int full_loop_enqueue(mpcb_handle *h, int cost_kind, int H, int64_t N, const double *init, const double *target,
                             const double *origin, const double *first_threshold, double eps, int max_ticks,
                             double *out_log, int32_t *out_ticks, int32_t *out_status, const mpcb_loop_trace &tr,
                             int *per_tick) {
    if (H < 1 || H > MPCB_MAX_H) return fail(h, MPCB_ERR_INVALID, "H=%d out of range [1,%d]", H, MPCB_MAX_H);
    if (cost_kind != MPCB_COST_MM && cost_kind != MPCB_COST_TREE) return fail(h, MPCB_ERR_INVALID, "bad mode/cost");
    CK(cudaSetDevice(h->device));
    int rc = ensure_tables(h);           // not inside a capture: it uploads from host vectors that die on return
    if (rc) return rc;
    CK(h->fl_state.ensure(sizeof(double) * 3 * N)); CK(h->fl_thr.ensure(sizeof(double) * N));
    CK(h->out_cost.ensure(sizeof(double) * N)); CK(h->out_index.ensure(sizeof(int64_t) * N));
    CK(h->out_traj.ensure(sizeof(double) * 3 * H * N)); CK(h->out_ctl.ensure(sizeof(double) * 2 * N));
    CK(h->fl_last.ensure(sizeof(double) * 5 * N));
    CK(h->fl_k.ensure(sizeof(int) * N)); CK(h->fl_have.ensure(sizeof(int) * N));
    CK(h->fl_flags.ensure(N)); CK(h->fl_count.ensure(2 * sizeof(int)));
    if (tr.pred) CK(h->fl_traj.ensure(sizeof(double) * N * 3 * H));
    FullLoopArgs fa{};
    fa.N = N; fa.H = H; fa.max_ticks = max_ticks; fa.eps = eps;
    fa.active_count = h->fl_count.as<int>(); fa.tick = fa.active_count + 1;
    fa.target = target;
    fa.best_cost = h->out_cost.as<double>(); fa.best_index = h->out_index.as<long long>();
    fa.best_traj = h->out_traj.as<double>(); fa.first_control = h->out_ctl.as<double>();
    fa.state = h->fl_state.as<double>(); fa.threshold = h->fl_thr.as<double>(); fa.last_ret = h->fl_last.as<double>();
    fa.kcount = h->fl_k.as<int>(); fa.have_ret = h->fl_have.as<int>(); fa.status = out_status;
    fa.ticks = out_ticks; fa.flags = h->fl_flags.as<unsigned char>();
    fa.log = out_log;
    fa.trace_pred = tr.pred; fa.trace_ctl = tr.control; fa.trace_cost = tr.cost;
    fa.last_traj = tr.pred ? h->fl_traj.as<double>() : nullptr;
    LoopGraphKey key;
    memset(&key, 0, sizeof key);
    key.epoch = h->epoch; key.N = N; key.cost_kind = cost_kind; key.H = H; key.max_ticks = max_ticks; key.eps = eps;
    const void *io[10] = {init, target, origin, first_threshold, out_log, out_ticks, out_status, tr.pred, tr.control, tr.cost};
    memcpy(key.io, io, sizeof io);
    key.allocs = g_allocs.load();
    if (h->fl_exec && !memcmp(&key, &h->fl_key, sizeof key)) {
        h->stats = h->fl_stats;
        *per_tick = h->fl_per_tick;
        return launch_loop_graph(h);
    }
    // solve_core's scratch grows outside the capture: a capture that needed a bigger buffer is dropped, the buffer
    // grown and the loop captured again (each round grows one more buffer; the sizes do not change between rounds)
    for (;;) {
        cudaGraph_t g = nullptr;
        CK(cudaGraphCreate(&g, 0));
        g_growth = DeferredGrowth{true, {}};
        rc = capture_full_loop(h, g, fa, cost_kind, init, origin, first_threshold, per_tick);
        g_growth.defer = false;
        const std::vector<std::pair<DevBuf *, size_t>> wanted = std::move(g_growth.wanted);
        g_growth.wanted.clear();
        if (rc == MPCB_OK) {
            cudaGraphExec_t exec = nullptr;
            const cudaError_t e = cudaGraphInstantiate(&exec, g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess)
                return fail(h, MPCB_ERR_CUDA, "full closed loop: graph instantiation failed: %s", cudaGetErrorString(e));
            if (h->fl_exec) h->fl_graphs.push_back(h->fl_exec);   // destroyed once the stream is idle
            key.allocs = g_allocs.load();      // the buffers grown for this capture are the ones it holds
            h->fl_key = key; h->fl_exec = exec;
            h->fl_stats = h->stats; h->fl_per_tick = *per_tick;
            return launch_loop_graph(h);
        }
        cudaGraphDestroy(g);
        if (wanted.empty()) return rc;
        for (const auto &w : wanted) CK(w.first->ensure(w.second));
    }
}

int mpcb_full_closed_loop_device(mpcb_handle *h, int cost_kind, int H, int64_t N, const double *init_state,
                                 const double *target, const double *origin, const double *first_threshold,
                                 double eps, int max_ticks, double *out_log, int32_t *out_ticks, int32_t *out_status) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (N < 0 || N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    if (N == 0) return MPCB_OK;
    if (!init_state || !target || !origin || !out_log || !out_ticks || !out_status || max_ticks < 1)
        return fail(h, MPCB_ERR_INVALID, "full closed loop: bad arguments");
    if (!h->have_grid) return fail(h, MPCB_ERR_NO_GRID, "mpcb_set_grid has not been called");
    int per_tick = 0;
    int rc = full_loop_enqueue(h, cost_kind, H, N, init_state, target, origin, first_threshold, eps, max_ticks, out_log,
                               out_ticks, out_status, tr, &per_tick);
    if (rc) return rc;
    h->stats.kernel_launches = per_tick;     // the tick count is known on the device only
    return MPCB_OK;
}

// host buffers -> device staging -> the loop graph -> host buffers, one synchronisation
int mpcb_full_closed_loop_host(mpcb_handle *h, int cost_kind, int H, int64_t N, const double *init_state,
                               const double *target, const double *origin, const double *first_threshold,
                               double eps, int max_ticks, double *out_log, int32_t *out_ticks, int32_t *out_status) {
    if (!h) return MPCB_ERR_INVALID;
    const mpcb_loop_trace tr = take_trace(h);
    if (N <= 0) return N == 0 ? MPCB_OK : fail(h, MPCB_ERR_INVALID, "N < 0");
    if (!init_state || !target || !origin || !out_log || !out_ticks || !out_status || max_ticks < 1)
        return fail(h, MPCB_ERR_INVALID, "full closed loop: bad arguments");
    if (!h->have_grid) return fail(h, MPCB_ERR_NO_GRID, "mpcb_set_grid has not been called");
    if (N >= (1LL << 31)) return fail(h, MPCB_ERR_INVALID, "N out of range");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const size_t nlog = (size_t)N * max_ticks * 5;
    CK(h->in_state.ensure(sizeof(double) * 3 * N)); CK(h->in_target.ensure(sizeof(double) * 2 * N));
    CK(h->in_origin.ensure(sizeof(double) * 2 * N));
    CK(h->loop_log.ensure(sizeof(double) * nlog)); CK(h->loop_ticks.ensure(sizeof(int) * N));
    CK(h->loop_status.ensure(sizeof(int) * N));
    CK(cudaMemcpyAsync(h->in_state.p, init_state, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_target.p, target, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->in_origin.p, origin, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    const double *d_thr = nullptr;
    if (first_threshold) {
        CK(h->in_thr.ensure(sizeof(double) * N));
        CK(cudaMemcpyAsync(h->in_thr.p, first_threshold, sizeof(double) * N, cudaMemcpyHostToDevice, st));
        d_thr = h->in_thr.as<double>();
    }
    CK(cudaMemsetAsync(h->loop_log.p, 0xFF, sizeof(double) * nlog, st));     // NaN pattern for unused rows
    const size_t nrow = (size_t)N * max_ticks;
    mpcb_loop_trace dtr{};
    int rc = stage_trace(h, tr, nrow, H, dtr);
    if (rc) return rc;
    int per_tick = 0;
    rc = full_loop_enqueue(h, cost_kind, H, N, h->in_state.as<double>(), h->in_target.as<double>(),
                           h->in_origin.as<double>(), d_thr, eps, max_ticks, h->loop_log.as<double>(),
                           h->loop_ticks.as<int>(), h->loop_status.as<int>(), dtr, &per_tick);
    if (rc) return rc;
    int ticks_run = 0;
    CK(cudaMemcpyAsync(&ticks_run, h->fl_count.as<int>() + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_log, h->loop_log.p, sizeof(double) * nlog, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_ticks, h->loop_ticks.p, sizeof(int) * N, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_status, h->loop_status.p, sizeof(int) * N, cudaMemcpyDeviceToHost, st));
    CK(copy_back_trace(h, tr, dtr, nrow, H));
    CK(cudaStreamSynchronize(st));
    retire_loop_graphs(h, true);
    h->stats.kernel_launches = ticks_run * per_tick;   // the solve's launches and the apply kernel, per tick run
    return MPCB_OK;
}

}  // extern "C"
