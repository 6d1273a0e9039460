// CUDA kernels (sm_100a) and the C ABI of include/mseetc_b200.h.
//
// Kernel roles (one lock-step "tick" = trial -> decide -> eval -> step):
//   k_cells<OP>  one thread per (interval k, instance): coalesced SoA streaming, HBM-bound
//   k_insts<OP>  one thread per instance: sequential sweeps over k (Riccati), loads coalesced across the warp
// No tensor cores: the per-interval blocks are 3x3 / 6x6 FP64 and there is no dense contraction.
#include <cuda_runtime.h>
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdio>
#include <limits>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/mseetc_b200.h"
#include "variants.h"
#include "compact.cuh"
#include "table.cuh"

using namespace mseetc;

static_assert((int)MSEETC_PARAM_COUNT == (int)PAR_N, "parameter plane enum out of sync");
static_assert((int)MSEETC_P_MASS == (int)P_MASS, "parameter plane enum out of sync");

namespace {

thread_local std::string g_err;


// ---- interval-parallel kernels: one thread per (interval k, instance), warp = 32 instances at one k.  The kernels stride over
// the cells, so any grid works; they are launched with one block per 128 cells (measured faster than a persistent grid of a few
// blocks per SM: 110.9k / 115.5k / 118.6k / 122.0k solves/s with 1/2/4/8 waves against 122.6k with the full grid on the bench
// workload).
// (MS_CELL_KERNEL: variants.h)
MS_CELL_KERNEL(k_cell_setup, 4, cell_setup(c, io, k, s))
MS_CELL_KERNEL(k_cell_init, 4, cell_init<false>(c, k, s))
// k_cell_trial_eval: the interval evaluation AT THE TRIAL POINT, which it forms on the way (one kernel per iteration instead of
// trial + evaluation); k_cell_eval: the same at the current iterate, once per solve for the starting point
MS_CELL_KERNEL(k_cell_trial_eval, 2, (cell_eval<false, true>(c, k, s)))
MS_CELL_KERNEL(k_cell_eval, 2, (cell_eval<false, false>(c, k, s)))
// (the variants with the spline loss map, the collocation integrator and integrated losses live in variants_*.cu: further translation units that
// compile next to this one, launched through mseetc::launch_variant)
MS_CELL_KERNEL(k_cell_step, CELL_STEP_MINB, cell_step<false>(c, k, s))
MS_CELL_KERNEL(k_cell_extract, 4, cell_extract(c, io, k, s))

__global__ void __launch_bounds__(64) k_inst_setup(Ctx c, BatchIO io) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < c.cfg.S) inst_setup(c, io, s);
}
// useSmem: dynamic shared memory holds two columns per thread (node speeds, interval lengths: 2 * NK * blockDim doubles)
__global__ void __launch_bounds__(128) k_inst_profile(Ctx c, int useSmem) {
    extern __shared__ double prof_sm[];
    // the first half of the block screens, the second half builds the starting profile of the same instances: the two walks
    // over the track are independent, so they run side by side (an instance that the screening flags gets a profile nobody reads)
    const int half = blockDim.x >> 1;
    const bool profileRole = (int)threadIdx.x >= half;
    const int col = profileRole ? (int)threadIdx.x - half : (int)threadIdx.x;
    const int s = blockIdx.x * half + col;
    if (s >= c.cfg.S) return;
    if (!profileRole) { inst_screen(c, s); return; }
    if (useSmem) inst_profile(c, s, prof_sm + col, prof_sm + (size_t)c.cfg.NK * half + col, half);
    else inst_profile(c, s);
}

// ---- per-instance reductions: one thread-block CLUSTER of RED_CL blocks per tile of 32 instances, RED_W warps in all; warp w sums
// the intervals k = w, w+RED_W, ... (coalesced rows) and the partials are combined in fixed order by warp 0 of the first block,
// which reads the other blocks' partials through distributed shared memory -> bitwise reproducible, no atomics.  A sweep of 2048
// running instances has only 64 tiles: one block per tile left 84 of the 148 SMs idle in these latency-bound kernels.
// `mirror` (mapped pinned host memory): the completion counter as it stands when this kernel runs, for the host's polling --
// a store from the kernel instead of a 4-byte cudaMemcpyAsync between two kernels of every tick (which cost ~10 us of stream time)
enum { RED_CL = 4, RED_WB = RED_W / RED_CL };      // blocks per cluster, warps per block
static_assert(RED_W % RED_CL == 0, "cluster size must divide the interleave factor");
__device__ __forceinline__ const double* cluster_peer(const double* p, unsigned rank) {
    return cooperative_groups::this_cluster().map_shared_rank(p, rank);
}
// The warp that runs the per-instance logic after the sums (filter test, convergence test, barrier update: a chain of dependent
// loads of the instance state) asks for that state just before the barrier (after its own share of the sums, which would flush it from L1), so that the chain finds it in L1 instead of paying
// one L2 round trip per link.
__device__ __forceinline__ void prefetch_instance_state(const Ctx& c, int s) {
    for (int f = 0; f < SD_N; ++f) asm volatile("prefetch.global.L1 [%0];" ::"l"(&c.D(f, s)));
    for (int f = 0; f < SI_N; ++f) asm volatile("prefetch.global.L1 [%0];" ::"l"(&c.I(f, s)));
}

__global__ void __cluster_dims__(RED_CL, 1, 1) __launch_bounds__(32 * RED_WB) k_inst_alpha(Ctx c, int* mirror) {
    namespace cg = cooperative_groups;
    cg::cluster_group cl = cg::this_cluster();
    if (mirror && blockIdx.x == 0 && threadIdx.x == 0) *mirror = *(volatile int*)c.done;
    __shared__ double sm[RED_WB][3][32];
    const unsigned rank = cl.block_rank();
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5, w = (int)rank * RED_WB + wl;
    const int s = (blockIdx.x / RED_CL) * 32 + lane;
    const bool on = s < c.cfg.nInst && c.I(SI_PHASE, s) == PH_STEPPED;
    double acc[3] = {1.0, 1.0, 0.0};
    if (on) alpha_partials(c, s, c.I(SI_N_INT, s), w, RED_W, acc);
    if (on && rank == 0 && wl == 0) prefetch_instance_state(c, s);
    for (int f = 0; f < 3; ++f) sm[wl][f][lane] = acc[f];
    cl.sync();
    double tot[3] = {1.0, 1.0, 0.0};
    if (rank == 0 && wl == 0 && on) {
        for (int ww = 0; ww < RED_W; ++ww) {
            const double* q = cluster_peer(&sm[ww % RED_WB][0][lane], ww / RED_WB);
            tot[0] = fmin(tot[0], q[0]); tot[1] = fmin(tot[1], q[32]); tot[2] += q[64];
        }
    }
    cl.sync();                                   // the peers' shared memory has been read: they may exit
    if (rank == 0 && wl == 0 && on) inst_alpha(c, s, tot);
}

// TRIAL = true: the sums belong to the trial point (in the other iterate buffer); the filter test (inst_decide) comes first and,
// when the point is accepted, the convergence test and the barrier update (inst_kkt) follow at once on the same sums.
// TRIAL = false: starting point, inst_kkt only.
template <bool TRIAL>
__global__ void __cluster_dims__(RED_CL, 1, 1) __launch_bounds__(32 * RED_WB) k_inst_kkt(Ctx c) {
    namespace cg = cooperative_groups;
    cg::cluster_group cl = cg::this_cluster();
    __shared__ double sm[RED_WB][10][32];      // field-major: conflict-free columns (one lane = one instance)
    const unsigned rank = cl.block_rank();
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5, w = (int)rank * RED_WB + wl;
    const int s = (blockIdx.x / RED_CL) * 32 + lane;
    const bool on = s < c.cfg.nInst && c.I(SI_PHASE, s) == (TRIAL ? PH_TRIAL : PH_EVAL);
    KktAcc acc;
    kkt_init(acc);
    if (on) kkt_partials(c, s, c.I(SI_N_INT, s), ((c.I(SI_PARITY, s) != 0) != TRIAL) ? WS_IT1 : WS_IT0, w, RED_W, acc);
    if (on && rank == 0 && wl == 0) prefetch_instance_state(c, s);
    sm[wl][0][lane] = acc.th; sm[wl][1][lane] = acc.fo; sm[wl][2][lane] = acc.slog; sm[wl][3][lane] = acc.sdamp;
    sm[wl][4][lane] = acc.zsum; sm[wl][5][lane] = acc.ysum; sm[wl][6][lane] = acc.dinf; sm[wl][7][lane] = acc.pinf;
    sm[wl][8][lane] = acc.cmin; sm[wl][9][lane] = acc.cmax;
    cl.sync();
    KktAcc tot;
    kkt_init(tot);
    const bool lead = rank == 0 && wl == 0 && on;
    if (lead) {
        for (int ww = 0; ww < RED_W; ++ww) {
            const double* q = cluster_peer(&sm[ww % RED_WB][0][lane], ww / RED_WB);
            KktAcc o;
            o.th = q[0]; o.fo = q[32]; o.slog = q[64]; o.sdamp = q[96];
            o.zsum = q[128]; o.ysum = q[160]; o.dinf = q[192]; o.pinf = q[224];
            o.cmin = q[256]; o.cmax = q[288];
            kkt_combine(tot, o);
        }
    }
    cl.sync();                                   // the peers' shared memory has been read: they may exit
    if (lead) {
        if (TRIAL) {
            const double sums[4] = {tot.th, tot.fo, tot.slog, tot.sdamp};
            inst_decide(c, s, sums);            // accepted: buffers swapped, phase -> evaluated
        } else count_cells(c, 4, c.I(SI_N_INT, s) + 1);
        inst_kkt(c, s, tot);                    // (nothing unless the point is the current iterate now)
    }
}

// Riccati sweeps: one thread per instance, stage data prefetched `depth` intervals ahead through a cp.async ring
// in dynamic shared memory ((depth+1) * RING_NF_MAX * blockDim doubles).
template <int BS, int DEPTH>
__global__ void __launch_bounds__(BS) k_step(Ctx c) {
    extern __shared__ __align__(128) double ring[];
    const int s = blockIdx.x * BS + threadIdx.x;
    if (s >= c.cfg.S) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool active = s < c.cfg.nInst && c.I(SI_PHASE, s) == PH_FACTOR;
    double* wring = ring + (size_t)warp * ((DEPTH + 1) * RING_NF_MAX * 32);
    if (!active) return;
    // every lane prefetches its own intervals (cp.async, one column per lane): works for mixed interval counts inside a tile
    RingFetch<BwdFields, 32, DEPTH> fb;
    fb.sm = wring + lane;
    RingFetch<FwdFields, 32, DEPTH> ff;
    ff.sm = wring + lane;
    inst_step(c, s, fb, ff);
}

// ---- parallel-in-time sweeps (pit.cuh): a block = SL consecutive instances x G chunk lanes, thread = (chunk l, instance).
// The lanes of a warp that work on the same chunk sit next to each other, so a warp touches 32/SL segments of SL * 8 bytes per
// field (whole 32-byte sectors for SL >= 4).  Elements, chunk-end values, chunk transitions and chunk-start states go through
// shared memory; the two short sequential chains over the chunks are run by the lane of chunk 0.  Stage data are prefetched
// through the same per-thread cp.async ring as in k_step.  An instance whose element algebra fails, or whose chain and recursion
// disagree, is redone by the sequential sweeps (lane of chunk 0, same kernel), so accuracy never rests on the chain.
// L2 prefetch distance of the sweep rings, in intervals beyond the ring's own look-ahead (none: 104 us, 3: 95 us)
enum { PIT_PF = 3 };
template <int SL, int G, int DEPTH>
__global__ void __launch_bounds__(SL * G) k_step_pit(Ctx c, int* fallbackCount) {
    extern __shared__ __align__(128) double pit_sm[];
    constexpr int BS = SL * G;
    double* ring = pit_sm;
    double* shbase = pit_sm + (size_t)(DEPTH + 1) * RING_NF_MAX * BS;
    int* flags = reinterpret_cast<int*>(shbase + (size_t)G * SH_N * SL);
    const int col = threadIdx.x % SL, l = threadIdx.x / SL;
    const int s = blockIdx.x * SL + col;
    const bool active = s < c.cfg.nInst && c.I(SI_PHASE, s) == PH_FACTOR;
    if (!__syncthreads_or(active)) return;
    PitShare sh{shbase, flags, SL};
    PitLane t;
    t.s = s; t.col = col; t.l = l; t.G = G;
    t.N = active ? c.I(SI_N_INT, s) : 2;
    t.mu = active ? c.D(SD_MU, s) : 0.1;
    t.delta = 0.0;
    const double dlast = active ? c.D(SD_DELTA_LAST, s) : 0.0;
    pit_chunk(t.N, G, l, t.kLo, t.kHi);
    if (active) pit_read_reference(c, t);
    if (l == 0) flags[col] = 0;
    RingFetch<BwdFields, BS, DEPTH, PIT_PF> fb;
    fb.sm = ring + threadIdx.x;
    // the forward sweep spends next to no arithmetic per interval: it needs the deeper look-ahead, and its 14 planes per interval
    // leave room for it in the same ring
    constexpr int FDEPTH = ((DEPTH + 1) * BwdFields::NF) / FwdFields::NF - 1;
    RingFetch<FwdFields, BS, FDEPTH, 2 * PIT_PF> ff;
    ff.sm = ring + threadIdx.x;
    double delta = 0.0;
    bool pending = active, failed = false, fallback = false;
    int why = 0;
    for (int tries = 0; tries < 40; ++tries) {
        // (this barrier also puts the reference reads and the flag reset before the first store of the pass)
        if (!__syncthreads_or(pending)) break;
        t.delta = delta;
        if (pending) {
            if (l == 0) count_cells(c, 2, t.N);
            pit_phase_a(c, t, sh, fb);
        }
        __syncthreads();
        if (pending && l == 0) pit_value_chain(sh, col, G);
        __syncthreads();
        if (pending) pit_phase_c(c, t, sh, fb);
        __syncthreads();
        const int f = flags[col];
        __syncthreads();
        if (l == 0) flags[col] = 0;
        if (pending) {
            if (f & PIT_SCAN_FAILED) { fallback = true; pending = false; why = f; }
            else if (f & PIT_BAD_INERTIA) {
                if (l == 0) c.I(SI_NREG, s) += 1;
                delta = pit_next_delta(delta, dlast);
                if (delta > 1e40) { failed = true; pending = false; }
            } else pending = false;
        }
    }
    if (pending) failed = true;
    if (__syncthreads_or(fallback)) {
        if (fallback && l == 0) {
            atomicAdd(fallbackCount, 1);
            if (why & PIT_ELEM_FAILED) atomicAdd(fallbackCount + 1, 1);
            if (why & PIT_APPLY_FAILED) atomicAdd(fallbackCount + 2, 1);
            if (why & PIT_INCONSISTENT) atomicAdd(fallbackCount + 3, 1);
            inst_step(c, s, fb, ff);            // complete sequential direction incl. its own inertia ladder and phase change
        }
        __syncthreads();
    }
    const bool go = active && !fallback && !failed;
    if (failed && l == 0) finish(c, s, ST_STEP_FAILED);
    if (go && l == 0) {
        pit_state_chain(sh, col, G);
        count_cells(c, 3, t.N);
        if (delta > 0.0) c.D(SD_DELTA_LAST, s) = delta;
        c.D(SD_DELTA, s) = delta;
    }
    __syncthreads();
    if (go) pit_phase_f(c, t, sh, ff);
    if (go && l == 0) { c.I(SI_FACT, s) = 1; c.I(SI_PHASE, s) = PH_STEPPED; }
}

// Loop condition of the device-side tick loop (CUDA graph conditional WHILE node): keep going while instances are running and the
// tick budget lasts.  ints of the counter block: [0] finished instances, [53] ticks done.
__global__ void k_loop_cond(cudaGraphConditionalHandle handle, int* counters, int n, int maxTicks) {
    const int tick = ++counters[53];
    cudaGraphSetConditional(handle, (*(volatile int*)counters < n && tick <= maxTicks) ? 1u : 0u);
}

__global__ void __launch_bounds__(128) k_cell_table(TableIO io, LossMapDev lm) {
    const size_t total = (size_t)(io.Nmax + 1) * io.n;
    for (size_t idx = (size_t)blockIdx.x * 128 + threadIdx.x; idx < total; idx += (size_t)gridDim.x * 128)
        cell_table(io, lm, (int)(idx % (io.Nmax + 1)), (int)(idx / (io.Nmax + 1)));
}
__global__ void __launch_bounds__(32) k_inst_resim(TableIO io) {
    inst_resim(io, blockIdx.x * 32 + threadIdx.x);
}

__global__ void k_eval_loss_rows(LossMapDev lm, int n, const double* in, const double* par, double* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    eval_loss_rows_point(lm, i, n, in, par, out);
}

// FP64 roofline denominator: 16 independent DFMA chains per thread, enough resident warps to keep the pipe full
__global__ void __launch_bounds__(256) k_fp64_peak(double* sink, int iters, double a, double b) {
    double x[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = a + 1e-3 * (threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = fma(x[i], b, a);
    }
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) acc += x[i];
    if (acc == 12345.678) sink[blockIdx.x * blockDim.x + threadIdx.x] = acc;      // never true: keeps the chains alive
}

__global__ void k_eval_interval(int n, int numSteps, int numApprox, const double* in, double* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    eval_interval_point<false>(i, n, numSteps, numApprox, in, out, nullptr);
}

}  // namespace

enum { CLS_TRIAL = 0, CLS_DECIDE, CLS_EVAL, CLS_STEP, CLS_MISC, CLS_CSTEP, CLS_ALPHA, CLS_KKT, NCLS };

struct mseetc_solver {
    mseetc_problem prob;
    int* done_host;     // pinned + mapped: [0] done counter, [16..] 4 x uint64 cell counters, [32..35] polling mirrors
    int* done_host_dev; // device alias of done_host
    int last_ticks;
    int last_launches;
    int profiling;
    double ms[NCLS];
    int launches[NCLS];
    long long cells[NCLS];
    std::vector<cudaEvent_t> ev;   // event pool (pairs), grown on demand, re-used across solves
    std::vector<int> ev_class;     // class of every event pair of the last solve (timeline)
    cudaEvent_t poll_ev[4];        // completion polling (see mseetc_solve_batch)
    int sweep_lanes;               // 0: chosen per call; 1: sequential sweeps; 8 / 16 / 32: chunk lanes per instance of the parallel-in-time sweeps
    int last_lanes;                // what the last solve used
    int last_compactions;          // compaction passes launched in the last solve
    int compaction;                // 1: compact the running batch (default)
    int last_moves;                // instances moved by the compaction passes of the last solve
    long long last_fallbacks;      // instances x iterations that fell back to the sequential sweeps in the last solve
    int fallback_why[3];           // of those: reference recursion failed / chain step singular / chain and recursion disagreed
    // device-side tick loop: a graph with one conditional WHILE node whose body is one tick, kept while the call's arguments repeat
    cudaGraph_t loop_graph;
    cudaGraphExec_t loop_exec;
    cudaStream_t cap_stream;
    int cap_prio;
    unsigned char loop_key[sizeof(Ctx) + sizeof(BatchIO) + 16];
    double* lm_dev;                // knots + coefficients of the dynamic loss map (loss_kind 2)
    LossMapDev lm;
    IrkTab* irk_dev;               // Butcher tableau of the collocation integrator in device memory; null: explicit RK4
    int int_losses;                // 1: integrateLosses = True (loss rows on integrated energies)
};

extern "C" {

int mseetc_version(void) { return MSEETC_B200_VERSION; }
const char* mseetc_last_error(void) { return g_err.c_str(); }

static int fail(int code, const char* msg) {
    g_err = msg;
    return code;
}
static int cuda_fail(cudaError_t e, const char* where) {
    g_err = std::string(where) + ": " + cudaGetErrorString(e);
    return (int)e;
}

int mseetc_create(const mseetc_problem* p, mseetc_handle* out) {
    if (!p || !out) return fail(-1, "mseetc_create: null argument");
    if (p->n_intervals_max < 2) return fail(-2, "mseetc_create: n_intervals_max must be >= 2");
    if (p->num_steps < 1 || p->num_approx_steps < 0) return fail(-3, "mseetc_create: bad RK options");
    if (p->loss_kind < 0 || p->loss_kind > 2) return fail(-4, "mseetc_create: loss_kind must be 0, 1 or 2");
    if (p->max_iterations < 1 || !(p->tol > 0.0) || !(p->mu_init > 0.0)) return fail(-5, "mseetc_create: bad IP options");
    if (p->initial_guess < 0 || p->initial_guess > 1) return fail(-7, "mseetc_create: initial_guess must be 0 or 1");
    mseetc_solver* h = new (std::nothrow) mseetc_solver;
    if (!h) return fail(-6, "mseetc_create: out of host memory");
    h->prob = *p;
    h->last_ticks = 0;
    h->last_launches = 0;
    h->profiling = 0;
    h->sweep_lanes = 1;
    h->last_lanes = 1;
    h->last_compactions = 0;
    h->last_fallbacks = 0;
    h->fallback_why[0] = h->fallback_why[1] = h->fallback_why[2] = 0;
    h->lm_dev = nullptr;
    h->irk_dev = nullptr;
    h->int_losses = 0;
    h->loop_graph = nullptr; h->loop_exec = nullptr; h->cap_stream = nullptr; h->cap_prio = 0;
    memset(h->loop_key, 0, sizeof h->loop_key);
    memset(&h->lm, 0, sizeof h->lm);
    for (int i = 0; i < NCLS; ++i) { h->ms[i] = 0.0; h->launches[i] = 0; h->cells[i] = 0; }
    cudaError_t e = cudaHostAlloc((void**)&h->done_host, 256, cudaHostAllocMapped);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaHostAlloc"); }
    e = cudaHostGetDevicePointer((void**)&h->done_host_dev, h->done_host, 0);
    if (e != cudaSuccess) { cudaFreeHost(h->done_host); delete h; return cuda_fail(e, "cudaHostGetDevicePointer"); }
    for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&h->poll_ev[i], cudaEventDisableTiming);
    if (e != cudaSuccess) { cudaFreeHost(h->done_host); delete h; return cuda_fail(e, "cudaEventCreateWithFlags"); }
    *out = h;
    return 0;
}

int mseetc_destroy(mseetc_handle h) {
    if (!h) return 0;
    cudaFreeHost(h->done_host);
    if (h->lm_dev) cudaFree(h->lm_dev);
    if (h->irk_dev) cudaFree(h->irk_dev);
    for (int i = 0; i < 4; ++i) cudaEventDestroy(h->poll_ev[i]);
    if (h->loop_exec) cudaGraphExecDestroy(h->loop_exec);
    if (h->loop_graph) cudaGraphDestroy(h->loop_graph);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    for (cudaEvent_t ev : h->ev) cudaEventDestroy(ev);
    delete h;
    return 0;
}

size_t mseetc_workspace_bytes(mseetc_handle h, int32_t n) {
    if (!h || n < 1) return 0;
    return plan_workspace(pad_slots(n), h->prob.n_intervals_max + 1).total;
}

int mseetc_last_ticks(mseetc_handle h) { return h ? h->last_ticks : -1; }
int mseetc_last_launches(mseetc_handle h) { return h ? h->last_launches : -1; }

int mseetc_set_loss_map(mseetc_handle h, int32_t nl, int32_t nv, const double* tl, const double* tv, const double* coef) {
    if (!h || !tl || !tv || !coef) return fail(-1, "mseetc_set_loss_map: null argument");
    if (nl < 4 || nv < 4) return fail(-2, "mseetc_set_loss_map: a cubic spline needs at least 4 coefficients per direction");
    const size_t count = (size_t)(nl + 4) + (nv + 4) + (size_t)nl * nv;
    if (h->lm_dev) { cudaFree(h->lm_dev); h->lm_dev = nullptr; }
    cudaError_t e = cudaMalloc((void**)&h->lm_dev, count * sizeof(double));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(loss map)");
    std::vector<double> host(count);
    memcpy(host.data(), tl, sizeof(double) * (nl + 4));
    memcpy(host.data() + nl + 4, tv, sizeof(double) * (nv + 4));
    memcpy(host.data() + nl + 4 + nv + 4, coef, sizeof(double) * (size_t)nl * nv);
    e = cudaMemcpy(h->lm_dev, host.data(), count * sizeof(double), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(loss map)");
    h->lm.tl = h->lm_dev; h->lm.tv = h->lm_dev + nl + 4; h->lm.coef = h->lm_dev + nl + 4 + nv + 4;
    h->lm.nl = nl; h->lm.nv = nv;
    return 0;
}

int mseetc_eval_loss_rows(mseetc_handle h, int32_t n, const double* in, const double* par, double* out, void* cuda_stream) {
    if (!h || n < 1 || !in || !par || !out) return fail(-1, "mseetc_eval_loss_rows: bad argument");
    if (!h->lm_dev) return fail(-2, "mseetc_eval_loss_rows: no loss map set (mseetc_set_loss_map)");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    k_eval_loss_rows<<<(n + 127) / 128, 128, 0, st>>>(h->lm, n, in, par, out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "k_eval_loss_rows launch");
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e, "k_eval_loss_rows");
    return 0;
}

int mseetc_set_sweep_lanes(mseetc_handle h, int lanes) {
    if (!h) return fail(-1, "mseetc_set_sweep_lanes: null handle");
    if (lanes != 0 && lanes != 1 && lanes != 8 && lanes != 16 && lanes != 32) return fail(-2, "mseetc_set_sweep_lanes: lanes must be 0 (auto), 1, 8, 16 or 32");
    h->sweep_lanes = lanes;
    return 0;
}
long long mseetc_last_sweep_fallbacks(mseetc_handle h) { return h ? h->last_fallbacks : -1; }
int mseetc_last_sweep_lanes(mseetc_handle h) { return h ? h->last_lanes : -1; }
int mseetc_last_compactions(mseetc_handle h) { return h ? h->last_compactions : -1; }
int mseetc_last_compaction_moves(mseetc_handle h) { return h ? h->last_moves : -1; }
int mseetc_set_compaction(mseetc_handle h, int on) {
    if (!h) return fail(-1, "mseetc_set_compaction: null handle");
    h->compaction = on ? 1 : 0;
    return 0;
}
int mseetc_last_sweep_fallback_reasons(mseetc_handle h, int32_t* out3) {
    if (!h || !out3) return fail(-1, "mseetc_last_sweep_fallback_reasons: null argument");
    for (int i = 0; i < 3; ++i) out3[i] = h->fallback_why[i];
    return 0;
}

int mseetc_set_integrate_losses(mseetc_handle h, int on) {
    if (!h) return fail(-1, "mseetc_set_integrate_losses: null handle");
    h->int_losses = on ? 1 : 0;
    memset(h->loop_key, 0, sizeof h->loop_key);
    return 0;
}

int mseetc_set_integrator(mseetc_handle h, int32_t stages, const double* A, const double* w, int32_t max_newton) {
    if (!h) return fail(-1, "mseetc_set_integrator: null handle");
    if (stages == 0) {                      // back to the explicit RK4 steps
        if (h->irk_dev) { cudaFree(h->irk_dev); h->irk_dev = nullptr; }
        memset(h->loop_key, 0, sizeof h->loop_key);
        return 0;
    }
    if (stages < 1 || stages > MS_IRK_MAXD || !A || !w || max_newton < 1) return fail(-2, "mseetc_set_integrator: 1 <= stages <= 9, tableau and max_newton >= 1 required");
    IrkTab t;
    memset(&t, 0, sizeof t);
    t.d = stages; t.maxNewton = max_newton;
    for (int i = 0; i < stages * stages; ++i) t.A[i] = A[i];
    for (int i = 0; i < stages; ++i) t.w[i] = w[i];
    cudaError_t e = cudaSuccess;
    if (!h->irk_dev) e = cudaMalloc((void**)&h->irk_dev, sizeof(IrkTab));
    if (e != cudaSuccess) { h->irk_dev = nullptr; return cuda_fail(e, "mseetc_set_integrator: cudaMalloc"); }
    e = cudaMemcpy(h->irk_dev, &t, sizeof t, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "mseetc_set_integrator: cudaMemcpy");
    return 0;
}

int mseetc_set_profiling(mseetc_handle h, int on) {
    if (!h) return fail(-1, "mseetc_set_profiling: null handle");
    h->profiling = on ? 1 : 0;
    return 0;
}

int mseetc_last_profile(mseetc_handle h, double* ms_out, int32_t* launches_out, int64_t* cells_out) {
    if (!h) return fail(-1, "mseetc_last_profile: null handle");
    for (int i = 0; i < NCLS; ++i) {
        if (ms_out) ms_out[i] = h->ms[i];
        if (launches_out) launches_out[i] = h->launches[i];
        if (cells_out) cells_out[i] = h->cells[i];
    }
    return 0;
}

// Algorithmic HBM traffic of one processed (interval, instance) cell, in bytes (FP64 planes read + written;
// per-instance scalars and parameters are warp-uniform broadcasts and not counted).  Derivation in DESIGN.md.
double mseetc_bytes_per_cell(mseetc_handle h, int cls) {
    if (!h) return 0.0;
    const mseetc_problem& p = h->prob;
    const int rows = (p.with_power_rows ? 2 : 0) + 1 + (p.energy_optimal ? 2 : 0);         // inequality rows
    const int nz = 2 + (p.with_pn_brake ? 2 : 0) + 1 + 4 + (p.with_power_rows ? 4 : 0) + 2 + (p.energy_optimal ? 2 : 0);
    const int prim = 4 + (p.with_pn_brake ? 1 : 0);
    const int iter = prim + rows + 2 + rows + nz;           // x, w, y, yd, z
    const int step = prim + rows + 2 + rows;
    const bool dynMap = (p.loss_kind == 2 && p.energy_optimal);
    switch (cls) {
        // evaluation at the trial point: reads iterate + step + 8 neighbour values + track 3, writes the trial iterate, the stage
        // QP and the partial sums
        case CLS_TRIAL:  return 8.0 * ((iter + step + 8 + 3) + iter + (QP_N - 2 * (NROW - rows) + 13)) - (dynMap ? 0.0 : 8.0 * 16);
        case CLS_DECIDE: return 8.0 * 14;
        case CLS_EVAL:   return 8.0 * ((iter + 4 + 3) + (QP_N - 2 * (NROW - rows) + 13)) - (dynMap ? 0.0 : 8.0 * 16);     // row gradients / residuals not stored
        // factors written: K 6, kf 2, P 6, p 3; the parallel-in-time sweeps read the condensed stage QP twice (element pass and
        // in-chunk recursion) -- the second read is counted: it is issued and, beyond L2, served by HBM
        case CLS_STEP:   return 8.0 * ((h->last_lanes > 1 ? 2 : 1) * BwdFields::NF + 17 + FwdFields::NF + 4);
        case CLS_CSTEP:  return 8.0 * ((6 + 3 + iter + 11 + rows + 2 + 7 + 6 + 9) + (2 * rows + 3 + 3)) - (dynMap ? 0.0 : 8.0 * 14);      // ... recomputed (+ b_{k+1}, c0)
        case CLS_ALPHA:  return 8.0 * 3;
        case CLS_KKT:    return 8.0 * 14;
        default:         return 0.0;
    }
}

int mseetc_solve_batch(mseetc_handle h, int32_t n, const double* params, const int32_t* nint, const int32_t* trk_of,
                       const int32_t* trk_off, const double* ds, const double* c0, const double* bmax, const double* tmin,
                       double* z_out,
                       double* lam_out, double* obj, double* kkt, int32_t* iters, int32_t* status, void* workspace,
                       size_t ws_bytes, void* cuda_stream) {
    if (!h) return fail(-1, "mseetc_solve_batch: null handle");
    if (n < 1) return fail(-2, "mseetc_solve_batch: n_instances must be >= 1");
    if (!params || !nint || !trk_of || !trk_off || !ds || !c0 || !bmax || !status || !workspace)
        return fail(-3, "mseetc_solve_batch: null device pointer");
    const mseetc_problem& p = h->prob;
    if (p.loss_kind == 2 && p.energy_optimal && !h->lm_dev) return fail(-6, "mseetc_solve_batch: loss_kind 2 needs mseetc_set_loss_map first");
    Config g;
    memset(&g, 0, sizeof g);
    g.S = pad_slots(n);
    g.NK = p.n_intervals_max + 1;
    g.nInst = n;
    g.withPn = p.with_pn_brake; g.withPower = p.with_power_rows; g.energy = p.energy_optimal; g.lossKind = p.loss_kind;
    g.numSteps = p.num_steps; g.numApprox = p.num_approx_steps; g.maxIter = p.max_iterations;
    g.tol = p.tol; g.muInit = p.mu_init; g.initMode = p.initial_guess; g.stallIters = p.stall_iterations;
    g.intLosses = (h->int_losses && p.energy_optimal) ? 1 : 0;
    WsPlan plan = plan_workspace(g.S, g.NK);
    if (ws_bytes < plan.total) return fail(-4, "mseetc_solve_batch: workspace too small (see mseetc_workspace_bytes)");
    if (((uintptr_t)workspace & 255) != 0) return fail(-5, "mseetc_solve_batch: workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    char* base = (char*)workspace;
    Ctx c;
    c.cfg = g;
    c.ws = (double*)(base + plan.off_ws);
    c.par = (double*)(base + plan.off_par);
    c.sd = (double*)(base + plan.off_sd);
    c.si = (int*)(base + plan.off_si);
    c.done = (int*)(base + plan.off_done);
    c.cnt = (unsigned long long*)(base + plan.off_done + 64);
    c.lm = h->lm;
    c.tmin = tmin;
    c.plan = (int*)(base + plan.off_plan);
    c.irk = h->irk_dev;
    const bool dyn = (p.loss_kind == 2 && p.energy_optimal);
    const bool intl = g.intLosses != 0;
    BatchIO io{params, nint, trk_of, trk_off, ds, c0, bmax, tmin, z_out, lam_out, obj, kkt, iters, status};

    const size_t cellThreads = (size_t)g.NK * g.S;
    const unsigned cgrid = (unsigned)((cellThreads + 127) / 128);      // grid of the interval kernels (see MS_CELL_KERNEL)
    const int ib = (g.S >= 148 * 64 * 2) ? 64 : 32;
    const unsigned igrid = (unsigned)((g.S + ib - 1) / ib);
    // prefetch depth of the Riccati ring: as deep as shared memory allows for the blocks resident on one SM
    int nsm = 148;
    {
        int devId = 0;
        cudaGetDevice(&devId);
        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, devId);
    }
    const int blocksPerSm = (int)((igrid + nsm - 1) / nsm);
    const size_t slotBytes = sizeof(double) * RING_NF_MAX * ib;
    int depth = (int)((size_t)200 * 1024 / ((size_t)(blocksPerSm < 1 ? 1 : blocksPerSm) * slotBytes)) - 1;
    // the depth is a compile-time constant of the kernel: largest instantiated value that fits
    void (*stepKernel)(Ctx);
    if (ib == 32) {
        // prefetch depth 16 measured slightly better than 8 (sweep launch 157 -> 153 us: the forward sweep spends ~0.15 us per
        // interval, so 8 intervals of look-ahead do not cover the DRAM latency under load)
        if (depth >= 16) { depth = 16; stepKernel = k_step<32, 16>; }
        else if (depth >= 8) { depth = 8; stepKernel = k_step<32, 8>; }
        else { depth = 4; stepKernel = k_step<32, 4>; }
    } else {
        if (depth >= 4) { depth = 4; stepKernel = k_step<64, 4>; }
        else if (depth >= 2) { depth = 2; stepKernel = k_step<64, 2>; }
        else { depth = 1; stepKernel = k_step<64, 1>; }
    }
    size_t ringBytes = (size_t)(depth + 1) * slotBytes;
    // The sweep blocks are spread over the SMs: the request is padded so that no more than blocksPerSm of them fit on one SM
    // (otherwise the block scheduler packs several of these one-warp, latency-bound blocks onto whatever SM has room while a
    // concurrent stream's interval kernels occupy the others, and they slow each other down: 243 -> 196 us per launch and
    // 129 k -> 137 k solves/s on the bench workload).
    {
        const int bps = blocksPerSm < 1 ? 1 : blocksPerSm;
        const size_t pad = (size_t)228 * 1024 / (bps + 1) + 1024;
        if (pad > ringBytes && pad <= (size_t)227 * 1024) ringBytes = pad;
    }
    // the attribute belongs to the kernel, not to this call: handles on other host threads launch the same kernel with other
    // sizes, so it is set to the hardware maximum rather than to this call's request
    cudaFuncSetAttribute(stepKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    // parallel-in-time sweeps: G = sweep_lanes chunk lanes per instance, SL instances per block.  Wider groups read longer
    // contiguous pieces of every plane (SL * 8 bytes): measured at 2048 active instances, 16 lanes: SL = 8 104 us, SL = 16 89 us
    // (4096 instances: 211 vs 148 us; 512 instances: 67 vs 76 us).  One instantiation per lane count, so that an instance gets
    // bit for bit the same direction whatever the size of the batch it is solved in.  Prefetch: one interval ahead through the
    // cp.async ring plus L2 prefetches three further on (a ring of depth 2 costs a resident block per SM: 124 vs 104 us).
    void (*pitKernel)(Ctx, int*) = nullptr;
    int pitThreads = 0, pitSL = 8;
    size_t pitBytes = 0;
    // 0 = auto: the sequential sweep is a dependent chain of n_intervals stages that takes the same time for 1 and for 4096
    // instances (153 us at 300 intervals); with G lanes the chain is ~2 n_intervals / G stages plus G - 2 short chain steps, at
    // 2.5 times the arithmetic and 1.4 times the bytes -- faster up to ~4096 instances per call (55 / 67 / 89 / 148 us at 32 /
    // 512 / 2048 / 4096 instances), slower beyond, where the sweeps are bandwidth-bound
    int lanesNow = h->sweep_lanes;
    if (lanesNow == 0) {
        const int Nmax = p.n_intervals_max;
        lanesNow = Nmax >= 1024 ? 32 : Nmax >= 96 ? 16 : Nmax >= 48 ? 8 : 1;
        if (lanesNow > 1 && lanesNow < 32 && g.S > 4096) lanesNow = 1;
    }
    h->last_lanes = lanesNow;
    if (lanesNow > 1) {
        const int G = lanesNow;
        pitSL = (G == 32) ? 8 : 16;
        if (G == 8) pitKernel = k_step_pit<16, 8, 1>;
        else if (G == 16) pitKernel = k_step_pit<16, 16, 1>;
        else pitKernel = k_step_pit<8, 32, 1>;
        pitThreads = pitSL * G;
        pitBytes = sizeof(double) * ((size_t)2 * RING_NF_MAX * pitThreads + (size_t)G * SH_N * pitSL) + sizeof(int) * pitSL;
        cudaFuncSetAttribute(pitKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    }
    int launches = 0;
    cudaError_t e;
    for (int i = 0; i < NCLS; ++i) { h->ms[i] = 0.0; h->launches[i] = 0; h->cells[i] = 0; }
    std::vector<int> evClass;   // class of each recorded event pair
    auto begin = [&](int cls) {
        h->launches[cls] += 1;
        ++launches;
        if (!h->profiling) return;
        const size_t need = 2 * (evClass.size() + 1);
        while (h->ev.size() < need) { cudaEvent_t x; cudaEventCreate(&x); h->ev.push_back(x); }
        cudaEventRecord(h->ev[2 * evClass.size()], st);
    };
    auto end = [&](int cls) {
        if (!h->profiling) return;
        cudaEventRecord(h->ev[2 * evClass.size() + 1], st);
        evClass.push_back(cls);
    };
    e = cudaMemsetAsync(c.done, 0, 256, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    e = cudaMemsetAsync(c.si, 0, sizeof(int) * (size_t)SI_N * g.S, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    const unsigned rgrid = (unsigned)(g.S / 32);
    begin(CLS_MISC); k_inst_setup<<<igrid, ib, 0, st>>>(c, io); end(CLS_MISC);
    begin(CLS_MISC); k_cell_setup<<<cgrid, 128, 0, st>>>(c, io); end(CLS_MISC);
    if (g.initMode || (tmin && g.energy)) {
        size_t profBytes = (size_t)2 * g.NK * ib * sizeof(double);
        if (profBytes > (size_t)200 * 1024 / (blocksPerSm < 1 ? 1 : blocksPerSm)) profBytes = 0;      // long horizons: scratch stays in HBM
        if (profBytes) cudaFuncSetAttribute(k_inst_profile, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        begin(CLS_MISC); k_inst_profile<<<igrid, 2 * ib, profBytes, st>>>(c, profBytes ? 1 : 0); end(CLS_MISC);
    }
    begin(CLS_MISC);
    if (intl) launch_variant(c.irk ? VK_INIT_INTL_IRK : VK_INIT_INTL, cgrid, st, c, io);
    else if (dyn) launch_variant(VK_INIT_DYN, cgrid, st, c, io); else k_cell_init<<<cgrid, 128, 0, st>>>(c, io);
    end(CLS_MISC);
    const int maxTicks = 3 * p.max_iterations + 100;
    int tick = 0;
    // ---- starting point: evaluation, convergence test, barrier parameter
    begin(CLS_EVAL);
    if (intl) launch_variant(c.irk ? VK_EVAL_INTL_IRK : VK_EVAL_INTL, cgrid, st, c, io);
    else if (c.irk) launch_variant(dyn ? VK_EVAL_DYN_IRK : VK_EVAL_IRK, cgrid, st, c, io);
    else if (dyn) launch_variant(VK_EVAL_DYN, cgrid, st, c, io); else k_cell_eval<<<cgrid, 128, 0, st>>>(c, io);
    end(CLS_EVAL);
    begin(CLS_KKT); k_inst_kkt<false><<<rgrid * RED_CL, 32 * RED_WB, 0, st>>>(c); end(CLS_KKT);
    // ---- the tick loop: direction (sweeps, interval-parallel rest, step-size limits), then the evaluation at the trial point with
    // the filter test / convergence test / barrier update: five launches per tick.
    // Small batches (latency): on the device -- a CUDA graph whose single node is a conditional WHILE node with one tick as its
    // body; the last kernel of the body sets the condition from the completion counter, so the host neither launches the ticks nor
    // polls.  Large batches keep the host loop below: it already runs two ticks ahead of the device, and next to the concurrent
    // minimum-time presolve (a second while-graph on a high-priority stream) the device loop measured slower (30.2 against 23.8 ms
    // per 4096-instance sweep).  Per-kernel profiling needs the host loop.
    h->last_compactions = 0;
    const bool useGraph = !h->profiling && g.S <= 256 && !tmin;
    auto tick_kernels = [&](cudaStream_t s0, int* mirror, bool prof) {
        if (prof) begin(CLS_STEP);
        if (pitKernel) pitKernel<<<(unsigned)(g.S / pitSL), pitThreads, pitBytes, s0>>>(c, c.done + 48);
        else stepKernel<<<igrid, ib, ringBytes, s0>>>(c);
        if (prof) end(CLS_STEP);
        if (prof) begin(CLS_CSTEP);
        if (intl) launch_variant(VK_STEP_INTL, cgrid, s0, c, io);
        else if (dyn) launch_variant(VK_STEP_DYN, cgrid, s0, c, io); else k_cell_step<<<cgrid, 128, 0, s0>>>(c, io);
        if (prof) end(CLS_CSTEP);
        if (prof) begin(CLS_ALPHA);
        k_inst_alpha<<<rgrid * RED_CL, 32 * RED_WB, 0, s0>>>(c, mirror);
        if (prof) end(CLS_ALPHA);
        if (prof) begin(CLS_TRIAL);
        if (intl) launch_variant(c.irk ? VK_TRIAL_INTL_IRK : VK_TRIAL_INTL, cgrid, s0, c, io);
        else if (c.irk) launch_variant(dyn ? VK_TRIAL_DYN_IRK : VK_TRIAL_IRK, cgrid, s0, c, io);
        else if (dyn) launch_variant(VK_TRIAL_DYN, cgrid, s0, c, io); else k_cell_trial_eval<<<cgrid, 128, 0, s0>>>(c, io);
        if (prof) end(CLS_TRIAL);
        if (prof) begin(CLS_DECIDE);
        k_inst_kkt<true><<<rgrid * RED_CL, 32 * RED_WB, 0, s0>>>(c);
        if (prof) end(CLS_DECIDE);
    };
    if (useGraph) {
        unsigned char key[sizeof h->loop_key];
        memset(key, 0, sizeof key);
        memcpy(key, &c, sizeof(Ctx));
        memcpy(key + sizeof(Ctx), &io, sizeof(BatchIO));
        int stPrio = 0;
        cudaStreamGetPriority(st, &stPrio);
        const int extra[4] = {lanesNow * 4 + (dyn ? 1 : 0), stPrio, maxTicks, n};
        memcpy(key + sizeof(Ctx) + sizeof(BatchIO), extra, sizeof extra);
        if (!h->loop_exec || memcmp(key, h->loop_key, sizeof key) != 0) {
            if (h->loop_exec) { cudaGraphExecDestroy(h->loop_exec); h->loop_exec = nullptr; }
            if (h->loop_graph) { cudaGraphDestroy(h->loop_graph); h->loop_graph = nullptr; }
            // the kernel nodes take the priority of the stream they are captured on: give the capture stream the priority of the
            // caller's stream
            if (h->cap_stream && stPrio != h->cap_prio) { cudaStreamDestroy(h->cap_stream); h->cap_stream = nullptr; }
            if (!h->cap_stream) {
                if ((e = cudaStreamCreateWithPriority(&h->cap_stream, cudaStreamNonBlocking, stPrio)) != cudaSuccess) return cuda_fail(e, "cudaStreamCreateWithPriority");
                h->cap_prio = stPrio;
            }
            if ((e = cudaGraphCreate(&h->loop_graph, 0)) != cudaSuccess) return cuda_fail(e, "cudaGraphCreate");
            cudaGraphConditionalHandle cond;
            if ((e = cudaGraphConditionalHandleCreate(&cond, h->loop_graph, 1, cudaGraphCondAssignDefault)) != cudaSuccess) return cuda_fail(e, "cudaGraphConditionalHandleCreate");
            cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
            np.conditional.handle = cond;
            np.conditional.type = cudaGraphCondTypeWhile;
            np.conditional.size = 1;
            cudaGraphNode_t node;
            if ((e = cudaGraphAddNode(&node, h->loop_graph, nullptr, 0, &np)) != cudaSuccess) return cuda_fail(e, "cudaGraphAddNode(conditional)");
            cudaGraph_t bodyGraph = np.conditional.phGraph_out[0];
            cudaStream_t cs = h->cap_stream;
            if ((e = cudaStreamBeginCaptureToGraph(cs, bodyGraph, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed)) != cudaSuccess) return cuda_fail(e, "cudaStreamBeginCaptureToGraph");
            tick_kernels(cs, nullptr, false);
            k_loop_cond<<<1, 1, 0, cs>>>(cond, c.done, n, maxTicks);
            cudaError_t le = cudaGetLastError();
            e = cudaStreamEndCapture(cs, nullptr);
            if (le != cudaSuccess) return cuda_fail(le, "tick capture");
            if (e != cudaSuccess) return cuda_fail(e, "cudaStreamEndCapture");
            if ((e = cudaGraphInstantiate(&h->loop_exec, h->loop_graph, 0)) != cudaSuccess) return cuda_fail(e, "cudaGraphInstantiate");
            memcpy(h->loop_key, key, sizeof key);
        }
        if ((e = cudaGraphLaunch(h->loop_exec, st)) != cudaSuccess) return cuda_fail(e, "cudaGraphLaunch");
    } else {
        for (;;) {
            // completion polling without draining the queue: k_inst_alpha mirrors the counter every tick into a small mapped
            // pinned ring and the mirror written two ticks ago is tested (its event has normally completed), so the kernels of
            // the next ticks are already queued
            tick_kernels(st, h->done_host_dev + 32 + tick % 4, true);
            ++tick;
            if (tick >= maxTicks) break;
            const int slot = (tick - 1) % 4;
            cudaEventRecord(h->poll_ev[slot], st);
            if (tick >= 3) {
                const int old = (tick - 3) % 4;
                e = cudaEventSynchronize(h->poll_ev[old]);
                if (e != cudaSuccess) return cuda_fail(e, "solver kernels");
                const int doneLag = h->done_host[32 + old];
                if (doneLag >= n) break;
                // compaction (compact.cuh): every fourth tick once instances have finished; the plan kernel decides on the device
                // whether the running instances are scattered enough to be worth moving, the other kernels return at once if not
                if (h->compaction &&!intl && g.S >= 256 && doneLag > 0 && tick % 4 == 0) {
                    const int activeUb = n - doneLag;
                    k_compact_plan<<<1, 1024, 0, st>>>(c);
                    k_compact_extract<<<cgrid, 128, 0, st>>>(c, io);
                    k_compact_move<<<(unsigned)(((size_t)activeUb * g.NK + 127) / 128), 128, 0, st>>>(c);
                    k_compact_finish<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(c);
                    k_compact_state<<<(unsigned)((activeUb + 127) / 128), 128, 0, st>>>(c);
                    launches += 5;
                    ++h->last_compactions;
                }
            }
        }
    }
    begin(CLS_MISC); k_cell_extract<<<cgrid, 128, 0, st>>>(c, io); end(CLS_MISC);
    if (intl && lam_out) launch_variant(c.irk ? VK_LAM_INTL_IRK : VK_LAM_INTL, cgrid, st, c, io);      // multipliers of the time rows in the reference's formulation
    e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
    e = cudaMemcpyAsync(h->done_host, c.done, 256, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(counters)");
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e, "solver kernels");
    {
        const unsigned long long* cnt = (const unsigned long long*)((const char*)h->done_host + 64);
        h->cells[CLS_TRIAL] = (long long)cnt[0];           // evaluations at trial points (accepted or not)
        h->cells[CLS_DECIDE] = (long long)cnt[0];
        h->cells[CLS_EVAL] = (long long)cnt[4];            // evaluation of the starting point
        h->cells[CLS_STEP] = (long long)cnt[1];
        h->cells[CLS_CSTEP] = (long long)cnt[3] + (long long)(cnt[3] / (unsigned long long)(p.n_intervals_max));
        h->cells[CLS_ALPHA] = h->cells[CLS_CSTEP];
        h->cells[CLS_KKT] = (long long)cnt[4];
        h->cells[CLS_MISC] = 0;
        h->last_fallbacks = (long long)h->done_host[48];
        for (int i = 0; i < 3; ++i) h->fallback_why[i] = h->done_host[49 + i];
    }
    for (size_t i = 0; i < evClass.size(); ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->ev[2 * i], h->ev[2 * i + 1]);
        h->ms[evClass[i]] += ms;
    }
    h->ev_class = evClass;
    if (useGraph) {
        tick = h->done_host[53];                      // ticks the device loop ran
        for (int cls : {CLS_STEP, CLS_CSTEP, CLS_ALPHA, CLS_TRIAL, CLS_DECIDE}) h->launches[cls] = tick;
        launches += 6 * tick;                         // five solver kernels and the loop condition per tick
    }
    h->last_ticks = tick;
    h->last_launches = launches;
    h->last_moves = h->done_host[54];
    return 0;
}

// Host-side preprocessing for many tracks at once (no pandas frame per track): the grid of computeDiscretizationPoints.
int mseetc_discretize_tracks(int32_t n_tracks, const double* length, const int32_t* n_int, const int32_t* lim_off, const double* lim_pos,
                             const double* lim_val, const int32_t* grd_off, const double* grd_pos, const double* grd_val, const int32_t* crv_off,
                             const double* crv_pos, const double* crv_val, const int32_t* out_off, double* pos_nodes, double* limit_nodes,
                             double* grad_nodes, double* curv_nodes, int32_t* error) {
    if (n_tracks < 1 || !length || !n_int || !lim_off || !lim_pos || !lim_val || !grd_off || !grd_pos || !grd_val || !crv_off || !crv_pos ||
        !crv_val || !out_off || !pos_nodes || !limit_nodes || !grad_nodes || !curv_nodes || !error)
        return fail(-1, "mseetc_discretize_tracks: bad argument");
    std::vector<double> brk, grid;
    for (int t = 0; t < n_tracks; ++t) {
        const int N = n_int[t];
        const double L = length[t];
        error[t] = 0;
        // merged section starts: outer join of the three step functions (track.py:377-383)
        brk.clear();
        brk.insert(brk.end(), lim_pos + lim_off[t], lim_pos + lim_off[t + 1]);
        brk.insert(brk.end(), grd_pos + grd_off[t], grd_pos + grd_off[t + 1]);
        brk.insert(brk.end(), crv_pos + crv_off[t], crv_pos + crv_off[t + 1]);
        std::sort(brk.begin(), brk.end());
        brk.erase(std::unique(brk.begin(), brk.end()), brk.end());
        const int M = (int)brk.size();
        const int nuni = N + 1 - (M - 1);                   // track.py:98
        if (N < 1 || nuni < 2) { error[t] = 1; continue; }
        grid.assign(brk.begin(), brk.end());
        const double step = L / (nuni - 1);
        for (int j = 0; j < nuni; ++j) grid.push_back(j == nuni - 1 ? L : j * step);        // numpy.linspace
        std::sort(grid.begin(), grid.end());
        grid.erase(std::unique(grid.begin(), grid.end()), grid.end());
        if ((int)grid.size() != N + 1) { error[t] = 1; continue; }                           // track.py:103-105
        double* po = pos_nodes + out_off[t] + t;
        double* lo = limit_nodes + out_off[t] + t;
        double* go = grad_nodes + out_off[t] + t;
        double* co = curv_nodes + out_off[t] + t;
        int il = lim_off[t], ig = grd_off[t], ic = crv_off[t];
        const double nan = std::numeric_limits<double>::quiet_NaN();
        for (int k = 0; k <= N; ++k) {                       // forward fill (track.py:101)
            const double x = grid[k];
            while (il + 1 < lim_off[t + 1] && lim_pos[il + 1] <= x) ++il;
            while (ig + 1 < grd_off[t + 1] && grd_pos[ig + 1] <= x) ++ig;
            while (ic + 1 < crv_off[t + 1] && crv_pos[ic + 1] <= x) ++ic;
            po[k] = x;
            lo[k] = (lim_off[t + 1] > lim_off[t] && lim_pos[il] <= x) ? lim_val[il] : nan;
            go[k] = (grd_off[t + 1] > grd_off[t] && grd_pos[ig] <= x) ? grd_val[ig] : nan;
            co[k] = (crv_off[t + 1] > crv_off[t] && crv_pos[ic] <= x) ? crv_val[ic] : nan;
        }
    }
    return 0;
}

int mseetc_table_columns(void) { return (int)TAB_NCOL; }

int mseetc_postprocess_batch(mseetc_handle h, int32_t n, const double* z, const double* params, const int32_t* nint, const int32_t* trk_of,
                             const int32_t* trk_off, const double* ds, const double* c0, const double* nodes, size_t node_stride,
                             const double* mass, const int32_t* status, double* table_out, void* cuda_stream) {
    if (!h) return fail(-1, "mseetc_postprocess_batch: null handle");
    if (n < 1) return fail(-2, "mseetc_postprocess_batch: n_instances must be >= 1");
    if (!z || !params || !nint || !trk_of || !trk_off || !ds || !c0 || !nodes || !mass || !table_out)
        return fail(-3, "mseetc_postprocess_batch: null device pointer");
    const mseetc_problem& p = h->prob;
    if (p.loss_kind == 2 && p.energy_optimal && !h->lm_dev) return fail(-6, "mseetc_postprocess_batch: loss_kind 2 needs mseetc_set_loss_map first");
    TableIO io{z, params, nint, trk_of, trk_off, ds, c0, nodes, node_stride, mass, status, table_out, n, p.n_intervals_max, p.with_pn_brake,
               p.energy_optimal ? p.loss_kind : 0};
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t total = (size_t)(io.Nmax + 1) * n;
    k_cell_table<<<(unsigned)((total + 127) / 128), 128, 0, st>>>(io, h->lm);
    k_inst_resim<<<(unsigned)((n + 31) / 32), 32, 0, st>>>(io);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "table kernels launch");
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e, "table kernels");
    return 0;
}

int mseetc_last_timeline(mseetc_handle h, mseetc_handle origin, double* out, int32_t max_entries) {
    if (!h || !origin || !out) return fail(-1, "mseetc_last_timeline: null argument");
    if (origin->ev_class.empty()) return 0;
    int n = 0;
    for (size_t i = 0; i < h->ev_class.size() && n < max_entries; ++i, ++n) {
        float a = 0.f, b = 0.f;
        if (cudaEventElapsedTime(&a, origin->ev[0], h->ev[2 * i]) != cudaSuccess) { cudaGetLastError(); break; }
        if (cudaEventElapsedTime(&b, origin->ev[0], h->ev[2 * i + 1]) != cudaSuccess) { cudaGetLastError(); break; }
        out[3 * n] = (double)h->ev_class[i]; out[3 * n + 1] = (double)a; out[3 * n + 2] = (double)b;
    }
    return n;
}

int mseetc_measure_fp64_peak(double* gflops_out, void* cuda_stream) {
    if (!gflops_out) return fail(-1, "mseetc_measure_fp64_peak: null argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = nsm * 8, threads = 256, iters = 20000;
    double* sink = nullptr;
    cudaError_t e = cudaMalloc((void**)&sink, sizeof(double) * (size_t)blocks * threads);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {        // first pass is the warm-up
        cudaEventRecord(a, st);
        k_fp64_peak<<<blocks, threads, 0, st>>>(sink, iters, 1.0000001, 0.9999999);
        cudaEventRecord(b, st);
        e = cudaEventSynchronize(b);
        if (e != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        const double gf = 2.0 * 16.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e9;
        if (rep > 0 && gf > best) best = gf;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(sink);
    if (e != cudaSuccess) return cuda_fail(e, "k_fp64_peak");
    *gflops_out = best;
    return 0;
}

int mseetc_eval_interval(int32_t n, int32_t num_steps, int32_t num_approx, const double* in, double* out, void* cuda_stream) {
    if (n < 1 || !in || !out) return fail(-1, "mseetc_eval_interval: bad argument");
    if (num_steps < 1 || num_approx < 0) return fail(-2, "mseetc_eval_interval: bad RK options");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    k_eval_interval<<<(n + 127) / 128, 128, 0, st>>>(n, num_steps, num_approx, in, out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "k_eval_interval launch");
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e, "k_eval_interval");
    return 0;
}

int mseetc_eval_interval_irk(int32_t n, int32_t num_steps, int32_t num_approx, int32_t stages, const double* A, const double* w,
                             int32_t max_newton, const double* in, double* out, void* cuda_stream) {
    if (n < 1 || !in || !out) return fail(-1, "mseetc_eval_interval_irk: bad argument");
    if (num_steps < 1 || num_approx < 0) return fail(-2, "mseetc_eval_interval_irk: bad step options");
    if (stages < 1 || stages > MS_IRK_MAXD || !A || !w || max_newton < 1) return fail(-3, "mseetc_eval_interval_irk: 1 <= stages <= 9, tableau and max_newton >= 1 required");
    IrkTab t;
    memset(&t, 0, sizeof t);
    t.d = stages; t.maxNewton = max_newton;
    for (int i = 0; i < stages * stages; ++i) t.A[i] = A[i];
    for (int i = 0; i < stages; ++i) t.w[i] = w[i];
    IrkTab* dev = nullptr;
    cudaError_t e = cudaMalloc((void**)&dev, sizeof t);
    if (e != cudaSuccess) return cuda_fail(e, "mseetc_eval_interval_irk: cudaMalloc");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    e = cudaMemcpyAsync(dev, &t, sizeof t, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        launch_eval_interval_irk(n, num_steps, num_approx, in, out, dev, st);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(dev);
    if (e != cudaSuccess) return cuda_fail(e, "k_eval_interval (irk)");
    return 0;
}

}  // extern "C"
