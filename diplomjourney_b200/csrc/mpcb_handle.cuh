// mpcb_handle.cuh -- the handle behind the C ABI (private to the library): one device, one stream, its growable
// device scratch.  Shared by mpcb_api.cu (solves) and mpcb_nccl.cu (cross-rank reconciliation).
#pragma once
#include <atomic>
#include <string>
#include <vector>

#include "mpcb_types.cuh"

namespace mpcb {

struct DevBuf;

// While the FULL closed loop captures its tick into a graph, no buffer may be freed or moved: the graph keeps the
// addresses it was captured with, and cudaFree cannot run during a capture.  With `defer` set, a buffer that would
// have to grow records the size wanted and ensure() fails; the loop grows the buffers after the capture and captures
// again (full_loop_enqueue, mpcb_api.cu).
struct DeferredGrowth {
    bool defer = false;
    std::vector<std::pair<DevBuf *, size_t>> wanted;
};
inline thread_local DeferredGrowth g_growth;

// Bumped whenever a buffer is (re)allocated: a cached FULL loop graph holds the addresses it was captured with.
inline std::atomic<unsigned long long> g_allocs{0};

// What a FULL loop graph froze at capture besides the handle's buffers (mpcb_api.cu, full_loop_enqueue); compared
// bytewise, so it is zeroed before it is filled.
struct LoopGraphKey {
    unsigned long long epoch, allocs;      // mpcb_handle_s::epoch, g_allocs
    long long N;
    int cost_kind, H, max_ticks;
    double eps;
    const void *io[10];                    // the caller's inputs, outputs and trace
};

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (g_growth.defer) {
            g_growth.wanted.emplace_back(this, bytes);
            return cudaErrorNotPermitted;
        }
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        g_allocs.fetch_add(1);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

constexpr unsigned long long kSegCap = 1ULL << 22;
constexpr unsigned long long kTileBatch = 1ULL << 23;   // subtree cut: tiles per batch (survivor list <= 64 MiB)
constexpr unsigned long long kWideReduceSegs = 1ULL << 15; // segments per solve from which the per-solve reduction runs grid-wide
constexpr unsigned long long kFrontierCap = 1ULL << 22; // frontier descent: entries per list (two lists = the tile list's 64 MiB)

}  // namespace mpcb

struct mpcb_handle_s {
    int device = 0, sms = 148;
    cudaStream_t stream = nullptr;
    std::string err;
    // grid
    bool have_grid = false, tables_ready = false;
    std::vector<double> hv, hb;         // host copy of the raw grids
    double L = 0, delta_t = 0, v_min = 0, v_slow = 0;
    mpcb::GridTables g{};
    mpcb::DevBuf tab64, tab32, vtab, tab64_slow, vtab_slow, beta, leaf32, leaf32p, leaf32r, ctl32, ctl32_slow;
    mpcb::RowPairs row_ab{};            // (a, b) of leaf32r's pairs: a kernel parameter of the exhaustive pass 1
    // options
    double tol_scale = 1.0;
    int algo = MPCB_ALGO_AUTO;
    int refine = 1;
    int small_path = 1;
    int zero_copy = 1;    // small_path with <= 64 solves: inputs and results in mapped pinned host memory, no copies
    int dump_direct = 0;  // mpcb_dump_leaves_host, prefix: dump the values pass 1 ranks with
    int npt = 4;          // exhaustive prefix pass 1: nodes per thread (profiles/r3f_stage1_ab.txt)
    unsigned long long frontier_cap = mpcb::kFrontierCap;   // entries per frontier list (option, diagnostics: a tiny value forces the fallback)
    int subtree_cut = 2;       // pruned pass 1, H >= 3: 0 off, 1 depth-(H-2) bound per 256-node tile, 2 auto (frontier descent from the root for trees of more than one tile batch), 3 frontier always
    int screen = 2;       // exhaustive prefix pass 1 (prune = 0): 2 = screen in two stages (distance first), 1 = screen loop without
                          // MUFU + rare full re-run, 0 = sqrt per leaf
    int prefilter = 1;    // pruned pass 1: fp32 pre-filter before the float64 node set-up (identical results)
    int prune = 1;        // exact branch-and-bound in the prefix kernel (identical results, fewer leaves evaluated)   // host-API HELD solves with few candidates take the one-launch float64 path
    // scratch
    mpcb::DevBuf sp, segmin, worklist, misc, tau, bestJ, bestIdx, lock, ub, tile_list, reduce_scratch;
    mpcb::DevBuf in_state, in_target, in_origin, in_thr, in_flags, out_cost, out_index, out_traj, out_ctl, dump_rec, dump_j;
    mpcb::DevBuf cand, cand_J, cand_sel;  // refinement: listed candidates, their float64 costs, per-solve (key, index)
    mpcb::DevBuf node_list;             // refinement: depth-(H-1) nodes whose leaves are to be scanned (RefineNode)
    unsigned node_cap = 1u << 15;       // entries of that list (option "node_list"; 0 = scan where found)
    unsigned cand_cap = 1u << 20;       // entries of that list (option "candidate_list"; 0 = evaluate where found)
    bool cand_auto = true;              // not set by the user: the prefix algorithm with a node list runs without it
    mpcb::DevBuf nccl_scratch;          // split tree: this rank's (cost, index) records + one slot per rank
    mpcb::DevBuf loop_log, loop_ticks, loop_status, loop_events, loop_final, loop_rng, loop_keys, loop_pcg, loop_pcg_spawn, small_in, small_out, fl_last, fl_k, fl_have, fl_flags, fl_count;
    mpcb::DevBuf fl_state, fl_thr;      // FULL loop: the robots' running poses and carried thresholds
    // FULL loop: the executable graph of the last call, launched again while its key holds, with the stats its capture
    // left and the kernels of one of its ticks; replaced graphs wait in fl_graphs until the stream is idle (destroying
    // an executable graph waits for the work in flight)
    unsigned long long epoch = 0;         // bumped by mpcb_set_grid and mpcb_set_option
    mpcb::LoopGraphKey fl_key{};
    cudaGraphExec_t fl_exec = nullptr;
    mpcb_stats fl_stats{};
    int fl_per_tick = 0;
    std::vector<cudaGraphExec_t> fl_graphs;
    mpcb_loop_trace trace{};            // of the next closed-loop call (mpcb_set_loop_trace), consumed by it
    mpcb::DevBuf trace_pred, trace_ctl, trace_cost, fl_traj;   // host entries: the trace staged on the device
    void *pin_in = nullptr, *pin_out = nullptr;   // pinned staging of the low-latency path
    size_t pin_in_cap = 0, pin_out_cap = 0;
    mpcb_stats stats{};
};
