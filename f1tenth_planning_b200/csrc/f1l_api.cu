// f1l_api.cu -- C-ABI (include/f1l.h) over the sm_100a kernels.  No torch types, no exceptions
// across the boundary; every launch goes on the handle's (or the caller's) stream.
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include <sched.h>
#include <unistd.h>

// NVTX ranges around the stages of the path (SURVEY 5: profiling hooks): sampler / eval / select
// launches, the H2D / D2H legs of the host-buffer calls.  Header-only NVTX3: a few tens of
// nanoseconds per call with no tool attached.
#include <nvtx3/nvToolsExt.h>
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

#include "f1l_common.cuh"
#include "f1l_lattice.cuh"
#include "f1l_peaks.cuh"
#include "f1l_pp.cuh"
#include "f1l_rollout.cuh"

#ifndef N_PIPE
#define N_PIPE 3  // streams of the host-buffer batch pipeline
#endif

namespace {

// An allocation the handle owns: freed by its destructor, i.e. at f1l_destroy's `delete h`, after
// the device synchronise.  DevBuf: device memory (grown by ensure); HostBuf: pinned host memory.
template <cudaError_t (*FREE)(void*)>
struct OwnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    OwnedBuf() = default;
    OwnedBuf(const OwnedBuf&) = delete;
    OwnedBuf& operator=(const OwnedBuf&) = delete;
    ~OwnedBuf() { reset(); }
    void reset() {
        if (p) FREE(p);
        p = nullptr;
        cap = 0;
    }
};
using DevBuf = OwnedBuf<cudaFree>;
using HostBuf = OwnedBuf<cudaFreeHost>;

// Per-scenario scratch of a sampler -> eval -> select pipeline: the sampler context, the goal
// centres, the argmin keys (which double as K1's key scratch) and K1's nearest points.  `best` has
// one 8-byte word behind the S keys: the persistent-grid work counter of a single query.
struct PipeScratch {
    DevBuf ctx, centres, best, near_i, near4;
    int reserve(f1l_handle h, int S);
};

// The per-scenario arrays of a host-buffer batch chunk, in the order they are copied
enum { B_POSES, B_OPP, B_NOPP, B_IDX, B_COST, B_TRAJ, B_COSTS, B_FLAGS, B_SS, B_PREV, B_PVALID, B_W, B_TERMS,
       B_VEL, B_ARRAYS };

struct PipeSlot {
    cudaStream_t stream = nullptr;
    PipeScratch scratch;
    DevBuf buf[B_ARRAYS];   // the chunk's device copies of those arrays
};

// A single query's choice of candidates as the caller gives it: the contiguous block
// [c_begin, c_end) (c_end <= 0: to the last), or with row_step > 1 the lookahead rows
// row0, row0 + row_step, ... of the goal grid
struct Shard {
    int c_begin = 0, c_end = 0, row0 = 0, row_step = 1;
};

// What a query covers, resolved (make_span): the evaluated shard-local candidates [c_begin, c_end),
// whose local index v maps to the candidate of lookahead row row0 + (v / nW) * row_step in the
// same column (row_step 1: v itself); the lookahead rows the sampler fills, s_row0 + k * s_step for
// k < s_rows; the candidate select returns when nothing at all was evaluated; and whether this rank
// evaluates nothing (it still takes part in the exchange, with key ~0).  All int: no padding,
// spans compare with memcmp.
struct Span {
    int C = 0;   // candidates per scenario
    int c_begin = 0, c_end = 0;
    int row0 = 0, row_step = 1;
    int s_row0 = 0, s_step = 1, s_rows = 0;
    int first = 0;
    int empty = 0;
};

}  // namespace

struct f1l_ctx {
    int device = 0;
    f1l_config cfg;
    cudaStream_t stream = nullptr;
    char err[512] = {0};
    int64_t launches = 0;
    int timing = 0;
    // CUDA graph of the single-query chain (H2D, sampler, eval, select, D2H)
    int use_graph = 1;
    unsigned long long epoch = 0;   // bumped by every upload / config change
    cudaGraphExec_t gexec = nullptr;
    unsigned long long gkey[2] = {~0ull, ~0ull};   // epoch and output mask of the captured graph
    double gvmin = 0.0;                            // ... v_min of a captured moving-opponent query
    Span gspan;                                    // ... and its span
    int timed = 0;  // events of the last pipeline launch are valid
#define F1L_EV_SLOTS 64
    cudaEvent_t ev[4 * F1L_EV_SLOTS] = {nullptr};
    int ev_next = 0, ev_count = 0;  // ring of (before sample, eval, select, after) event quads
    float last_ms[3] = {0, 0, 0};
    int sm_count = 148;
    // track
    int n = 0, ncols = 0;
    DevBuf xy, v, psi, kappa, segA, segB, blk;
    DevBuf seg_s;      // [n-1] double2 (cumulative length at the segment's start, length): rollout progress
    double lap = 0.0;  // cumulative length of the n-1 segments plus the closing gap p_{n-1} -> p_0
    // grid
    DevBuf grid, clear, clear_tmp, edt;
    int use_clearance = 1;
    int gh = 0, gw = 0;
    double gox = 0, goy = 0, gres = 1;
    // lut
    DevBuf lut;
    int ldims[3] = {20, 21, 9};
    double lranges[6] = {0.2, 4.0, -2.0, 2.0, -1.5707963267948966, 1.5707963267948966};
    // goal grid
    DevBuf lookaheads, widths;
    int nL = 0, nW = 0;
    // previous path
    DevBuf prev;
    int has_prev = 0, prev_m = 0;
    // single-query device buffers
    PipeScratch q_scratch;
    DevBuf q_in, q_goals, q_states, q_headings, q_params, q_flags;
    // pinned staging for the single query
    HostBuf h_in;   // pose + opponents
    HostBuf h_out;  // result block (QHeader | best trajectory | map-frame trajectory)
    void* h_out_dev = nullptr;  // the same block as the device sees it (mapped pinned memory): the
                                // select kernel of a single query writes its results straight into it
    // per-candidate detail block of a single query (costs | terms | goals | params | flags): one
    // device block, one D2H into pinned staging, then plain copies into the caller's arrays
    DevBuf q_detail;
    HostBuf h_detail;
    // deviation-pass work counters (f1l_set_stats / f1l_get_stats)
    DevBuf stats;
    int stats_on = 0;
    // batch (device-pointer API) scratch, also the scratch of every rollout step
    PipeScratch b_scratch;
    // rollout (f1l_rollout_dev) scratch: command, cost, the races' opponent table
    DevBuf r_ss, r_cost, r_opp, r_nopp;
    DevBuf r_vel;   // the races' opponent velocities [S,F1L_MAX_OPP,2] (f1l_rollout_predict_dev)
    DevBuf mo_dbg;  // k_t and (wx, wy) of the last moving-opponent single query (f1l_debug_motion_ctx)
    // batch pipeline (host-pointer API)
    PipeSlot pipe[N_PIPE];
    // device copies of the arrays of the one-shot host-buffer calls (pure pursuit, intersect, ...)
    DevBuf m[7];
    DevBuf pp_key;   // K1's key scratch of the pure-pursuit / front-axle device calls
    // peer-memory exchange of candidate-sharded queries (f1l_xchg_*): the local block, the peers'
    // blocks as mapped by cudaIpcOpenMemHandle (own rank: the local pointer)
    int pp_per_sm = 0, pp_per_sm_ct = 0;   // resident pp_scan_kernel CTAs per SM (pp_slots): global / constant table
    unsigned long long ctab_key = 0;   // != 0: this handle's track sits in the constant-memory table
                                       // (as long as it is still the device's owner, ctab_owner)
    DevBuf xchg;
    XchgView xview = {0, 0, {nullptr}};
    // template instance / CTA plan of the last eval_kernel launch (f1l_last_eval_shape)
    int eval_info[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    // the last single query, for f1l_select_candidate: its span, explicit goals?, epoch
    Span lastq_span;
    int lastq_goals = 0;
    unsigned long long lastq_epoch = ~0ull;
};

namespace {

int fail(f1l_handle h, cudaError_t e, const char* what) {
    if (h) snprintf(h->err, sizeof(h->err), "%s: %s", what, cudaGetErrorString(e));
    return F1L_ERR_CUDA;
}

#define CK(call)                                            \
    do {                                                    \
        cudaError_t e__ = (call);                           \
        if (e__ != cudaSuccess) return fail(h, e__, #call); \
    } while (0)

int ensure(f1l_handle h, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap && b.p) return F1L_OK;
    // a captured single-query graph bakes device pointers in: any (re)allocation invalidates it
    h->epoch++;
    if (b.p) {
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes < 256 ? 256 : bytes;
    CK(cudaMalloc(&b.p, want));
    b.cap = want;
    return F1L_OK;
}

#define ENS(buf, bytes)                          \
    do {                                         \
        int r__ = ensure(h, (buf), (bytes));     \
        if (r__ != F1L_OK) return r__;           \
    } while (0)

int PipeScratch::reserve(f1l_handle h, int S) {
    ENS(ctx, sizeof(QueryCtx) * (size_t)S);
    ENS(centres, sizeof(Centre) * (size_t)S * (h->nL > 0 ? h->nL : 1));
    ENS(best, 8 * (size_t)S + 8);
    ENS(near_i, 4 * (size_t)S);
    ENS(near4, 32 * (size_t)S);
    return F1L_OK;
}

// One per-item host array of a host-buffer call and its device copy.  A null source and
// destination: the call has no such array, and the device sees a null pointer.
struct Stage {
    DevBuf* buf;
    const void* src;   // copied in (nullable)
    void* dst;         // copied back (nullable)
    size_t bytes;      // per item
    void* dev() const { return src || dst ? buf->p : nullptr; }
};

// ensures the device copies of items [i0, i0 + n), then enqueues the inputs' H2D copies
template <int K>
int stage_in(f1l_handle h, cudaStream_t st, const Stage (&t)[K], size_t i0, size_t n) {
    for (const Stage& e : t)
        if (e.src || e.dst) ENS(*e.buf, n * e.bytes);
    for (const Stage& e : t)
        if (e.src)
            CK(cudaMemcpyAsync(e.buf->p, (const char*)e.src + i0 * e.bytes, n * e.bytes, cudaMemcpyHostToDevice, st));
    return F1L_OK;
}

// enqueues the outputs' D2H copies of items [i0, i0 + n)
template <int K>
int stage_out(f1l_handle h, cudaStream_t st, const Stage (&t)[K], size_t i0, size_t n) {
    for (const Stage& e : t)
        if (e.dst)
            CK(cudaMemcpyAsync((char*)e.dst + i0 * e.bytes, e.buf->p, n * e.bytes, cudaMemcpyDeviceToHost, st));
    return F1L_OK;
}

// explicit goals [C,3] f64 -> float4 (x, y, theta, 0) in q_goals, by way of the caller's `g4`
// (which must outlive the copy)
int upload_goals(f1l_handle h, const double* goals, int C, std::vector<float>& g4, cudaStream_t st) {
    g4.assign(4 * (size_t)C, 0.0f);
    for (size_t c = 0; c < (size_t)C; ++c) {
        g4[4 * c] = (float)goals[3 * c];
        g4[4 * c + 1] = (float)goals[3 * c + 1];
        g4[4 * c + 2] = (float)goals[3 * c + 2];
    }
    ENS(h->q_goals, (size_t)C * 16);
    CK(cudaMemcpyAsync(h->q_goals.p, g4.data(), (size_t)C * 16, cudaMemcpyHostToDevice, st));
    return F1L_OK;
}

TrackView track_view(f1l_handle h) {
    TrackView t;
    t.n = h->n;
    t.ncols = h->ncols;
    t.xy = (const double2*)h->xy.p;
    t.v = (const double*)h->v.p;
    t.psi = (const double*)h->psi.p;
    t.kappa = (const double*)h->kappa.p;
    t.segA = (const float4*)h->segA.p;
    t.segB = (const float2*)h->segB.p;
    t.blk_origin = (const double2*)h->blk.p;
    return t;
}

GridView grid_view(f1l_handle h) {
    GridView g;
    g.occ = (const uint8_t*)h->grid.p;
    // three covering discs (collision_mode 1): centres -L/3, 0, +L/3 on the body axis, radius
    // sqrt((L/6)^2 + (W/2)^2); thresholds on the squared cell distance of the transform
    const double L = h->cfg.car_length, W = h->cfg.car_width;
    const double r_cells = std::sqrt(L * L / 36.0 + W * W / 4.0) / h->gres;
    const double off_cells = (L / 3.0) / h->gres;
    g.edt2 = (const uint16_t*)h->edt.p;
    // centre-to-centre cell distances: the disc centre lies within half a cell diagonal of its
    // cell's centre and an occupied cell reaches half a diagonal beyond its own, so the discs
    // (hence the rectangle they cover) are clear of every occupied cell iff d > r + sqrt(2)
    const double t = r_cells + 1.4142135623730951;
    g.disc_t2 = (int)std::floor(t * t) + 1;
    g.disc_off = (float)(L / 3.0);
    if (h->cfg.collision_mode == 1) {
        // the outer discs' cells lie within off + sqrt(2) (+1 for FP32 cell rounding) cells of the
        // centre's cell and the transform is 1-Lipschitz: at this distance no disc can collide
        const double far = std::sqrt((double)g.disc_t2) + off_cells + 2.5;
        g.near_map = g.edt2;
        g.near_free = (int)std::ceil(far * far);
    } else {
        // all nine probes fall within ceil(r_circ / res) cells of the centre cell (+1 for
        // rounding): a larger Chebyshev clearance proves them free
        const double rc = 0.5 * std::sqrt(L * L + W * W);
        const int probe_reach = (int)std::ceil(rc / h->gres) + 1;
        g.near_map = h->use_clearance ? (const uint16_t*)h->clear.p : nullptr;
        g.near_free = probe_reach + 1;
        if (probe_reach > CLEAR_R) g.near_map = nullptr;   // map too fine for the clearance radius
    }
    g.h = h->gh;
    g.w = h->gw;
    g.ox = h->gox;
    g.oy = h->goy;
    g.inv_res = 1.0 / h->gres;
    return g;
}

LutView lut_view(f1l_handle h) {
    LutView l;
    l.cells = (const float4*)h->lut.p;
    l.nx = h->ldims[0];
    l.ny = h->ldims[1];
    l.nt = h->ldims[2];
    l.x0 = (float)h->lranges[0];
    l.y0 = (float)h->lranges[2];
    l.t0 = (float)h->lranges[4];
    l.sx = l.nx > 1 ? (float)((l.nx - 1) / (h->lranges[1] - h->lranges[0])) : 0.0f;
    l.sy = l.ny > 1 ? (float)((l.ny - 1) / (h->lranges[3] - h->lranges[2])) : 0.0f;
    l.st = l.nt > 1 ? (float)((l.nt - 1) / (h->lranges[5] - h->lranges[4])) : 0.0f;
    return l;
}

EvalParams eval_params(f1l_handle h) {
    const f1l_config& c = h->cfg;
    EvalParams e;
    e.M = c.n_samples;
    e.n_newton = c.n_newton;
    e.window = c.window;
    e.n_shift = c.n_shift;
    e.n_cull = c.n_cull;
    e.literal_tracker = c.literal_tracker;
    e.use_goal_kappa = c.use_goal_kappa;
    e.generator = c.generator;
    e.prune = c.prune_window != 0;
    e.collision_mode = c.collision_mode;
    for (int i = 0; i < F1L_N_TERMS; ++i) e.w[i] = (float)c.weights[i];
    e.kappa_max = (float)c.kappa_max;
    e.half_l = (float)(0.5 * c.car_length);
    e.half_w = (float)(0.5 * c.car_width);
    const double hl = 0.5 * c.car_length, hw = 0.5 * c.car_width;
    e.rc2 = (float)(4.0 * (hl * hl + hw * hw));
    e.reach_pad = sqrtf(e.rc2) + 1e-3f;
    e.inv_M = 1.0f / (float)c.n_samples;
    e.tol = (float)c.converge_tol;
    e.tracker_lookahead = c.tracker_lookahead;
    e.wheelbase = c.wheelbase;
    e.max_reacquire = c.max_reacquire;
    return e;
}

int check_config(const f1l_config* c) {
    if (!c) return F1L_ERR_INVALID_ARG;
    if (c->n_samples < 2 || c->n_samples > F1L_MAX_M) return F1L_ERR_INVALID_ARG;
    if (c->n_newton < 0 || c->n_newton > 64) return F1L_ERR_INVALID_ARG;
    if (c->n_shift < 0 || c->n_cull < 0) return F1L_ERR_INVALID_ARG;
    if (c->generator < 0 || c->generator > 1) return F1L_ERR_INVALID_ARG;
    if (c->collision_mode < 0 || c->collision_mode > 1) return F1L_ERR_INVALID_ARG;
    if (!(c->car_length > 0) || !(c->car_width > 0)) return F1L_ERR_INVALID_ARG;
    return F1L_OK;
}

// ---- kernel instances per sample count ---------------------------------------------------------
typedef void (*eval_fn)(EvalArgs);
typedef void (*select_fn)(SelectArgs);
typedef void (*generate_fn)(LutView, EvalParams, const float4*, int, float4*, float4*, uint8_t*);

// dynamic shared memory an eval_kernel launch may use: the opt-in maximum is 227 KB per block
// INCLUDING static shared memory
constexpr int EVAL_SMEM_MAX = 226 * 1024;

// One compiled eval_kernel: the resident CTAs per SM its register budget is built for (MINB), and
// its shared memory in front of the window table (EvalSmem::C_TAB).
// shared memory the MO twin stages in front of the window table (the opponent velocities and k_t)
constexpr uint32_t EVAL_MO_SMEM = EvalSmem<1, 8, 1, true>::C_TAB - EvalSmem<1, 8, 1>::C_TAB;

struct EvalBuild {
    eval_fn fn;     // null: not built
    eval_fn fn_w;   // the same with per-scenario cost weights (null: not built)
    int minb;
    uint32_t smem_fixed;
    eval_fn fn_m = nullptr;   // fn_w's twin with moving opponents (null: not built)
    size_t smem_bytes(int nseg_pad, bool mo = false) const {
        return smem_fixed + (mo ? EVAL_MO_SMEM : 0) + (size_t)(nseg_pad + EVAL_SEG_PAD) * (2 * sizeof(float4));
    }
};

// The kernels that serve sample counts M <= m_max: the deviation-pass shape (IPL samples per lane;
// S samples per lane x SG sample groups in the loop), one eval build per warp count, and the select
// and generate kernels of the same IPL.
struct EvalBucket {
    int m_max, ipl, s, sg;
    EvalBuild nw4, nw7, nw8;
    EvalBuild wide;   // 8 warps at two CTAs per SM (128 registers), large dense queries (no
                      // per-scenario weights: lone queries plan with the config's)
    select_fn select;
    generate_fn generate;
    const EvalBuild& build(int nw) const { return nw == 4 ? nw4 : (nw == 7 ? nw7 : nw8); }
};

template <int IPL, int S, int SG, int NW, int MINB, bool WEIGHTS = true>
EvalBuild eval_build() {
    if constexpr (MINB == 0) return {nullptr, nullptr, 0, 0};
    else if constexpr (!WEIGHTS) return {eval_kernel<IPL, S, SG, NW, MINB, false>, nullptr, MINB, EvalSmem<S, SG, NW>::C_TAB};
    else return {eval_kernel<IPL, S, SG, NW, MINB, false>, eval_kernel<IPL, S, SG, NW, MINB, true>, MINB,
                 EvalSmem<S, SG, NW>::C_TAB, eval_kernel<IPL, S, SG, NW, MINB, true, true>};
}
template <int M_MAX, int IPL, int S, int SG, int MINB4, int MINB7, int MINB8, int MINB_WIDE>
EvalBucket eval_bucket() {
    return {M_MAX, IPL, S, SG,
            eval_build<IPL, S, SG, 4, MINB4>(), eval_build<IPL, S, SG, 7, MINB7>(),
            eval_build<IPL, S, SG, 8, MINB8>(), eval_build<IPL, S, SG, 8, MINB_WIDE, false>(),
            select_kernel<IPL>, generate_kernel<IPL>};
}

// Every eval_kernel instance and its residency, one row per bucket (MINB 0: no such build).
// NW = 7 (four resident CTAs of 7 warps at <= 72 registers) serves candidate counts that are a
// small multiple of 7 -- the default 4x7 goal grid; everything else runs 8-warp CTAs (three at 80).
// The M > 128 shapes have no 4- and 7-warp builds: their 72-register builds spill, so the launch
// policy only ever runs them on 8 warps.
// The M <= 104 shape on 4-warp CTAs (the batch regime of the 4x7 grid) runs FOUR CTAs per SM at
// 125 registers instead of seven at 72 -- the deviation loop gets the schedule it wants (no spill,
// 8.2 instead of 9.6 sub-partition cycles per (sample, segment) in isolation) and sixteen warps per
// SM still cover the latency-bound stages: 11.10 -> 10.84 ms on the bench workload (five CTAs at
// 96 registers: 11.16, six at 80: 11.26, three at 161: 11.69; S = 7 x SG = 16 instead of 13 x 8:
// 11.53; profiles/r2_microbench.md).  The wide build of the M > 128 shapes, two 8-warp CTAs per SM
// at 128 registers, gives the deviation loop the registers it wants
// (tools/microbench/devloop_bench.cu) at the price of a third fewer resident warps: it pays for a
// dense query with many candidates per warp slot (the unsharded 65 536), not for its shards.
//
//                  M <=  IPL   S  SG   MINB at NW = 4, 7, 8, 8 (wide)
const EvalBucket kEvalBuckets[] = {
    eval_bucket<      32,   1,  4,  8,   7, 4, 3, 0>(),
    eval_bucket<      64,   2,  8,  8,   7, 4, 3, 0>(),
    eval_bucket<     104,   4, 13,  8,   4, 4, 3, 0>(),
    eval_bucket<     128,   4, 16,  8,   7, 4, 3, 0>(),
    eval_bucket<     208,   7, 13, 16,   0, 0, 3, 2>(),
    eval_bucket<F1L_MAX_M,  8, 16, 16,   0, 0, 3, 2>(),
};

const EvalBucket& eval_bucket_of(int M) {
    for (const EvalBucket& b : kEvalBuckets)
        if (M <= b.m_max) return b;
    return kEvalBuckets[sizeof(kEvalBuckets) / sizeof(kEvalBuckets[0]) - 1];
}

// CTA plan of the eval kernel: NW warps per CTA, `chunk` candidates per CTA.  NW = 7 runs four
// resident CTAs per SM (72 registers, 28 warps), NW = 8 three (80 registers, 24 warps); besides
// exact divisibility (no idle warp in the last round of a CTA) the choice minimises the number
// of CTA waves, which is what decides the latency of one dense query.
constexpr int EVAL_ITEM = 4;   // candidates a warp takes at a time to share their Newton solves
struct CtaPlan {
    int nw, chunk, ctas_per_scn;
};

CtaPlan plan_ctas(int n_cand, int S, int M, int sm_count, bool cubic) {
    CtaPlan best{8, 8, 1};
    double best_cost = 1e300;
    // Throughput regime -- many waves of small scenarios (the 4x7 grid: 28 candidates) with shared
    // Newton solves: one 4-warp CTA per scenario whose warps pull the scenario's 4-candidate items.
    // Measured, not modelled (the wave model below counts CTAs and would always prefer the CTA with
    // more warps at equal residency): 10.84 ms on the bench workload against 11.19 for 7-warp CTAs.
    const EvalBucket& bucket = eval_bucket_of(M);
    {
        const int full4 = ((n_cand + 3) / 4) * 4;
        if (cubic && bucket.nw4.fn && full4 >= 4 * EVAL_ITEM && n_cand <= 256 &&
            (long long)S >= 8LL * bucket.nw4.minb * sm_count)
            return CtaPlan{4, full4, 1};
    }
    const int nws[3] = {4, 7, 8};
    for (int nw : nws) {
        if (!bucket.build(nw).fn) continue;
        const int resident = bucket.build(nw).minb * sm_count;
        const int full = ((n_cand + nw - 1) / nw) * nw;   // one CTA per scenario
        // chunk sizes worth a look: enough CTAs for ~8 waves (dense single queries), the smallest
        // chunk whose warps share Newton solves, and the whole scenario in one CTA
        long long per = (8LL * resident + S - 1) / S;
        const long long max_per = (n_cand + nw - 1) / nw;
        if (per > max_per) per = max_per;
        if (per < 1) per = 1;
        int c8 = (int)((n_cand + per - 1) / per);
        c8 = ((c8 + nw - 1) / nw) * nw;
        const int options[3] = {c8, EVAL_ITEM * nw < full ? EVAL_ITEM * nw : full, full};
        for (int chunk : options) {
            const int cps = (n_cand + chunk - 1) / chunk;
            const double ctas = (double)S * cps;
            const double waves = std::ceil(ctas / resident);
            // candidates a warp runs one after the other; with the cubic generator and at least four
            // candidates per warp they are taken four at a time (shared Newton solve)
            const int item = (cubic && chunk >= 4 * nw) ? EVAL_ITEM : 1;
            const double rounds = std::ceil(std::ceil((double)chunk / item) / nw) * item;
            // time ~ waves x (rounds + prologue) + tail, in units of one candidate per warp: a
            // candidate whose Newton solve is not shared costs ~6 % more instructions, the CTA
            // prologue (window table, set-up) ~0.3 candidates, and the last wave's CTAs hold their
            // SMs until their slowest warps finish: about half a candidate.  Slightly favour the
            // configuration with more resident warps on ties.
            double cost = (waves * (rounds * (item == EVAL_ITEM ? 1.0 : 1.06) + 0.3) + 0.5) * (nw == 7 ? 0.999 : 1.0);
            // Throughput regime (many waves of whole-scenario CTAs sharing Newton solves): measured
            // on the 10^5 x 28 batch, seven 4-warp CTAs per SM whose warps pull the scenario's seven
            // items (2 + 2 + 2 + 1) beat four 7-warp CTAs with one item per warp by 0.8 % -- the
            // once-per-warp set-up runs in 4 instead of 7 warps and idle warp slots turn over in
            // smaller units -- although the round count says otherwise (8 against 4 per CTA).
            if (nw == 4 && item == EVAL_ITEM && waves >= 8 && cps == 1) cost *= 0.9;
            if (cost < best_cost) { best_cost = cost; best = {nw, chunk, cps}; }
        }
    }
    return best;
}

// The eval_kernel instance one pipeline launch runs, and its CTA plan
struct EvalChoice {
    const EvalBucket* bucket;
    const EvalBuild* build;
    int nw, chunk, ctas_per_scn, item;
    bool persistent;   // one wave of CTAs pulling candidates from a device-wide counter
    bool wide;         // build is bucket->wide
    bool pw;           // per-scenario cost weights: build->fn_w
    bool mo;           // moving opponents: build->fn_m (pw is set too)
    eval_fn fn() const { return mo ? build->fn_m : (pw ? build->fn_w : build->fn); }
};

// The whole instance choice of a pipeline launch (launch_pipeline, f1l_debug_eval_choice): the CTA
// plan, the persistent grid and the wide build of a lone dense query, and the PW twin of a call
// with per-scenario cost weights.  lone: a single query with a persistent-grid counter and a
// non-empty span.  motion: the MO twin of the PW instance, chosen as for a call with weights.
EvalChoice choose_eval(int n_cand, int S, int M, int sm_count, bool cubic, bool lone, bool weights,
                       bool motion = false) {
    weights = weights || motion;
    const CtaPlan cp = plan_ctas(n_cand, S, M, sm_count, cubic);
    EvalChoice c;
    c.bucket = &eval_bucket_of(M);
    c.build = &c.bucket->build(cp.nw);
    c.nw = cp.nw;
    c.chunk = cp.chunk;
    c.ctas_per_scn = cp.ctas_per_scn;
    // four candidates per warp at a time (shared Newton) when every warp has at least four
    c.item = (cubic && cp.chunk >= 4 * cp.nw) ? EVAL_ITEM : 1;
    c.pw = weights;
    c.mo = motion;
    // A lone dense query that needs more than one wave of CTAs runs on a PERSISTENT grid instead: one
    // wave of CTAs whose warps pull single candidates from a device-wide counter, far lookahead rows
    // (the expensive candidates) first.  No wave quantisation, one window-table prologue per
    // resident CTA, and the cheap early-exit candidates fill the tail.
    long long resident = (long long)c.build->minb * sm_count;
    c.persistent = lone && cp.nw != 4 && cp.ctas_per_scn > resident;
    // ... and with at least EVAL_WIDE_MIN candidates per resident warp it runs the 128-register
    // build of the M > 128 shapes on two CTAs per SM (measured on config 5: 65 536 candidates
    // 471 -> 431 us, 32 768: 247 -> 234, 16 384: 134 -> 128, 8 192: 76 -> 100)
    constexpr int EVAL_WIDE_MIN = 4;
    c.wide = c.persistent && cp.nw == 8 && c.bucket->wide.fn && !weights &&
             (long long)n_cand >= EVAL_WIDE_MIN * resident * cp.nw;
    if (c.wide) {
        c.build = &c.bucket->wide;
        resident = (long long)c.build->minb * sm_count;
    }
    if (c.persistent) {
        // single candidates per pull, unless every warp has at least four 4-candidate items to go
        // through: then the shared Newton solve pays more than the coarser tail costs
        c.item = (cubic && (long long)n_cand >= 16LL * resident * cp.nw) ? EVAL_ITEM : 1;
        if (c.ctas_per_scn > resident) c.ctas_per_scn = (int)resident;
    }
    return c;
}

// owner of the constant-memory line-form table of each device (f1l_pp.cuh): the key of the handle
// whose f1l_set_track filled it last
// (host threads: a scan that uses the table is enqueued under g_ctab_mu after re-checking the
// owner, and an upload first withdraws the ownership under the same mutex, then drains the device,
// then writes -- so no enqueued scan can meet another track's entries)
static unsigned long long g_ctab_owner[64] = {0};
static unsigned long long g_ctab_serial = 0;
static std::mutex g_ctab_mu;
bool ctab_valid(f1l_handle h) {
    return h->ctab_key != 0 && h->device >= 0 && h->device < 64 && g_ctab_owner[h->device] == h->ctab_key;
}

// resident one-warp scan CTAs on the handle's device, from the occupancy calculator (once)
int pp_slots(f1l_handle h) {
    const bool ct = ctab_valid(h);
    int& per_sm = ct ? h->pp_per_sm_ct : h->pp_per_sm;
    if (per_sm <= 0) {
        int n = 0;
        const cudaError_t e = ct ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, pp_scan_kernel<true>, 32, 0)
                                 : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, pp_scan_kernel<false>, 32, 0);
        if (e != cudaSuccess || n <= 0) n = PP_TASK_MINB;
        per_sm = n;
    }
    return per_sm * h->sm_count;
}

// K1 = key preset + scan + finish on one stream over the handle's track.  key: 8 bytes of scratch
// per pose
void launch_pp(f1l_handle h, cudaStream_t stream, const double* poses, int pose_stride, int n_poses,
               double L, double wb, double max_reacquire, int front_axle, double k_path,
               unsigned long long* key, const PPOut& o) {
    const TrackView tv = track_view(h);
    bool ctab = ctab_valid(h);
    const int n_groups = (n_poses + PP_CTA_POSES - 1) / PP_CTA_POSES;
    const int nblk = (tv.n - 1 + 31) >> 5;
    const int n_parts = pp_task_parts(n_groups, nblk, pp_slots(h), ctab ? 16 : 6);
    cudaMemsetAsync(key, 0xff, (size_t)n_poses * 8, stream);
    PPParts parts;
    parts.n = n_parts;
    parts.per = nblk / n_parts;
    parts.rem = nblk - parts.per * n_parts;
    const dim3 grid((unsigned)n_groups, (unsigned)n_parts);
    if (ctab) {
        std::lock_guard<std::mutex> lk(g_ctab_mu);
        ctab = ctab_valid(h);   // still ours?  (checked and enqueued under the mutex)
        if (ctab)
            pp_scan_kernel<true><<<grid, 32, 0, stream>>>(tv, poses, pose_stride, n_poses, front_axle, wb, parts, key);
    }
    if (!ctab)
        pp_scan_kernel<false><<<grid, 32, 0, stream>>>(tv, poses, pose_stride, n_poses, front_axle, wb, parts, key);
    pp_finish_kernel<<<(n_poses + PP_THREADS - 1) / PP_THREADS, PP_THREADS, 0, stream>>>(
        tv, poses, pose_stride, n_poses, L, wb, max_reacquire, front_axle, k_path, key, o);
}

struct BatchOut {
    int32_t* best_idx = nullptr;
    float* best_cost = nullptr;
    int32_t* status = nullptr;
    double* steer_speed = nullptr;
    float4* best_traj = nullptr;
    double* best_traj_map = nullptr;   // [S,M,4] map frame (X, Y, v, Theta)
    float* costs = nullptr;
    float* terms = nullptr;
    uint8_t* flags = nullptr;
    float* goals_out = nullptr;
    float4* params = nullptr;
    float4* states = nullptr;
    float2* headings = nullptr;
    float* prev_out = nullptr;         // [S,M] theta column of each best trajectory (update_prev)
    uint8_t* prev_valid_out = nullptr; // [S] set to 1 with it (per-scenario previous paths)
    int32_t* xchg_status = nullptr;    // sharded single query: != 0 when a peer did not arrive
};

// Inputs of a pipeline over S scenarios: device pointers (host ones in a host-buffer batch call)
struct PipeIn {
    const double* poses = nullptr;     // [S,4]
    const double* opp = nullptr;       // [S,max_opp,3] (null: no opponents)
    const int32_t* n_opp = nullptr;    // [S] (null: max_opp each)
    int S = 0, max_opp = 0;
    const float4* goals = nullptr;     // [span.C] explicit goals (null: the goal grid)
    Span span;
    // previous paths: scenario s reads prev_theta + s * prev_stride (stride 0: one path for all)
    // when prev_valid is null or prev_valid[s] != 0; prev_theta null: no similarity term
    const float* prev_theta = nullptr;
    int prev_stride = 0;
    const uint8_t* prev_valid = nullptr;
    const float* weights = nullptr;    // [S,5] cost weights per scenario (null: the config's)
    const XchgView* xc = nullptr;      // sharded single query: exchange the argmin with the peers
    int* work_next = nullptr;          // single query: device counter for the persistent-grid schedule
    // moving opponents: velocities [S,max_opp,2] (null without opponents), the ego's v_min
    bool motion = false;
    const double* opp_vel = nullptr;
    double v_min = 1.0;
    float* mo_ctx = nullptr;           // debug copy of scenario 0's k_t and velocities (nullable)
};

// The span of a query over the explicit goals (n_goals > 0) or the goal grid (n_goals 0), with the
// peers' exchange taking place or not: every check of the candidate and row arguments
int make_span(f1l_handle h, int n_goals, const Shard& q, bool exchange, Span& sp) {
    sp = Span{};
    sp.C = n_goals > 0 ? n_goals : h->nL * h->nW;
    if (sp.C <= 0) return F1L_ERR_NO_GOALS;
    sp.s_rows = h->nL;
    if (q.row_step > 1) {   // row-interleaved shard: rows row0, row0 + row_step, ... of the goal grid
        if (n_goals > 0 || q.row0 < 0 || q.row0 >= q.row_step) return F1L_ERR_INVALID_ARG;
        const int n_rows = q.row0 < h->nL ? (h->nL - q.row0 + q.row_step - 1) / q.row_step : 0;
        // More ranks than lookahead rows: with peers attached the call is collective, so a rank
        // without rows must still arrive at the exchange (it contributes key = ~0 and returns the
        // global winner like everybody else); alone there is nothing to answer.
        if (n_rows == 0) {
            if (!exchange) return F1L_ERR_INVALID_ARG;
            sp.empty = 1;
        }
        sp.c_end = n_rows * h->nW;
        sp.row0 = q.row0;
        sp.row_step = sp.s_step = q.row_step;
        sp.s_row0 = sp.empty ? 0 : q.row0;   // the sampler fills this shard's rows only
        sp.s_rows = n_rows;
        sp.first = sp.empty ? 0 : q.row0 * h->nW;
        return F1L_OK;
    }
    sp.c_begin = q.c_begin > 0 ? q.c_begin : 0;
    sp.c_end = q.c_end > 0 && q.c_end < sp.C ? q.c_end : sp.C;
    if (sp.c_begin >= sp.c_end) return F1L_ERR_INVALID_ARG;
    sp.first = sp.c_begin;
    if (n_goals == 0 && (sp.c_begin > 0 || sp.c_end < sp.C)) {
        // contiguous candidate block: the lookahead rows it touches
        sp.s_row0 = sp.c_begin / h->nW;
        sp.s_rows = (sp.c_end - 1) / h->nW - sp.s_row0 + 1;
    }
    return F1L_OK;
}

// select_kernel arguments of a pipeline
SelectArgs select_args(f1l_handle h, const PipeIn& in, const PipeScratch& sc, const BatchOut& o) {
    SelectArgs se;
    if (in.xc && in.S == 1) se.xc = *in.xc;
    else { se.xc.world = 0; se.xc.rank = 0; }
    se.xchg_status = o.xchg_status;
    se.tr = track_view(h);
    se.lut = lut_view(h);
    se.ep = eval_params(h);
    se.ctx = (const QueryCtx*)sc.ctx.p;
    se.centres = (const Centre*)sc.centres.p;
    se.widths = (const float*)h->widths.p;
    se.nL = h->nL;
    se.nW = h->nW;
    se.inv_nW = 1.0f / (float)(h->nW > 0 ? h->nW : 1);
    se.row0 = in.span.s_row0;
    se.row_step = in.span.s_step;
    se.n_rows = in.span.s_rows;
    se.goals = in.goals;
    se.C = in.span.C;
    se.c_begin = in.span.first;
    se.best = (const unsigned long long*)sc.best.p;
    se.best_idx = o.best_idx;
    se.best_cost = o.best_cost;
    se.status = o.status;
    se.steer_speed = o.steer_speed;
    se.best_traj = o.best_traj;
    se.best_traj_map = o.best_traj_map;
    se.prev_theta_out = o.prev_out;
    se.prev_valid_out = o.prev_valid_out;
    return se;
}

// sampler -> eval -> select on `stream`, with `sc` reserved for in.S scenarios
int launch_pipeline(f1l_handle h, cudaStream_t stream, const PipeIn& in, PipeScratch& sc,
                    const BatchOut& o, bool time_it) {
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    const int S = in.S;
    const Span& sp = in.span;
    if (in.max_opp > F1L_MAX_OPP || in.max_opp < 0) return F1L_ERR_INVALID_ARG;
    QueryCtx* ctx = (QueryCtx*)sc.ctx.p;
    Centre* centres = (Centre*)sc.centres.p;
    unsigned long long* best = (unsigned long long*)sc.best.p;
    const int M = h->cfg.n_samples;
    const EvalParams ep = eval_params(h);
    if (ep.collision_mode == 1 && h->grid.p) {
        // the distance transform is exact up to CLEAR_R cells: a finer map needs a larger radius
        const GridView gv = grid_view(h);
        if (gv.near_free > CLEAR_R * CLEAR_R) return F1L_ERR_TOO_LARGE;
    }
    const int nsegs = h->n - 1;
    int nseg = h->cfg.window;
    if (nseg <= 0 || nseg > nsegs) nseg = nsegs;
    const int nseg_pad = (nseg + 31) & ~31;
    const int n_cand = sp.empty ? 1 : sp.c_end - sp.c_begin;
    const EvalChoice ec = choose_eval(n_cand, S, M, h->sm_count, ep.generator == 0,
                                      S == 1 && in.work_next && !sp.empty, in.weights != nullptr, in.motion);
    if (!ec.fn()) return F1L_ERR_INVALID_ARG;   // the choice names an instance that is not built
    const bool dyn = ec.persistent;
    const size_t smem = ec.build->smem_bytes(nseg_pad, ec.mo);
    if (smem > EVAL_SMEM_MAX) return F1L_ERR_TOO_LARGE;

    SampleArgs sa;
    sa.tr = track_view(h);
    sa.grid = grid_view(h);
    sa.ep = ep;
    sa.poses = in.poses;
    sa.opp = in.opp;
    sa.n_opp = in.n_opp;
    sa.max_opp = in.max_opp;
    sa.lookaheads = (const double*)h->lookaheads.p;
    sa.nL = in.goals ? 0 : h->nL;
    sa.row0 = sp.s_row0;
    sa.row_step = sp.s_step;
    sa.n_rows = sp.s_rows;
    sa.ctx = ctx;
    sa.centres = centres;
    sa.best = best;
    sa.work_next = dyn ? in.work_next : nullptr;
    cudaEvent_t* ev = h->ev + 4 * h->ev_next;
    if (time_it) cudaEventRecord(ev[0], stream);
    nvtxRangePushA("f1l.sample");
    if (S >= 32) {
        // batch: nearest_point of all scenarios by the thread-per-pose scan kernel (K1), then one
        // warp per scenario for the lookahead intersections / context
        PPOut po{};
        po.nearest = (double*)sc.near4.p;
        po.nearest_i = (int32_t*)sc.near_i.p;
        launch_pp(h, stream, in.poses, 4, S, -1.0, 0.33, 0.0, 0, 0.0, best, po);   // `best` doubles as K1's key scratch: the sampler resets it
        sample_warp_kernel<<<(S + SAMPLE_WARPS - 1) / SAMPLE_WARPS, SAMPLE_WARPS * 32, 0, stream>>>(
            sa, po.nearest_i, po.nearest, S);
        h->launches += 2;
    } else {
        // a lone dense query: one warp per ~2 lookahead rows; small batches: 8 warps each
        int st_threads = SAMPLE_THREADS;
        if (S <= 4 && sa.n_rows > 8) {
            st_threads = ((sa.n_rows + 1) / 2) * 32;
            if (st_threads > SAMPLE_THREADS_MAX) st_threads = SAMPLE_THREADS_MAX;
            if (st_threads < SAMPLE_THREADS) st_threads = SAMPLE_THREADS;
        }
        sample_kernel<<<S, st_threads, 0, stream>>>(sa);
    }
    nvtxRangePop();
    if (time_it) cudaEventRecord(ev[1], stream);

    NvtxRange nvtx_eval_select("f1l.eval+select");
    EvalArgs ea;
    ea.tr = sa.tr;
    ea.grid = sa.grid;
    ea.lut = lut_view(h);
    ea.ep = ep;
    ea.ctx = ctx;
    ea.centres = centres;
    ea.widths = (const float*)h->widths.p;
    ea.nL = h->nL;
    ea.nW = h->nW;
    ea.goals = in.goals;
    ea.prev_theta = in.prev_theta;
    ea.prev_stride = in.prev_stride;
    ea.prev_valid = in.prev_valid;
    ea.weights = in.weights;
    ea.C = sp.C;
    ea.c_begin = sp.c_begin;
    ea.c_end = sp.c_end;
    ea.row0 = sp.row0;
    ea.row_step = sp.row_step;
    ea.chunk = ec.chunk;
    ea.ctas_per_scn = ec.ctas_per_scn;
    ea.item = ec.item;
    ea.work_next = dyn ? in.work_next : nullptr;
    ea.v_last = dyn ? sp.c_begin + sp.c_end - 1 : 0;
    ea.inv_nW = 1.0f / (float)(h->nW > 0 ? h->nW : 1);
    ea.nseg_pad = nseg_pad;
    ea.costs = o.costs;
    ea.terms = o.terms;
    ea.flags = o.flags;
    ea.goals_out = o.goals_out;
    ea.params = o.params;
    ea.states = o.states;
    ea.headings = o.headings;
    ea.best = best;
    ea.stats = h->stats_on ? (unsigned long long*)h->stats.p : nullptr;
    ea.opp_vel = in.motion ? in.opp_vel : nullptr;
    ea.vel_stride = in.max_opp;
    ea.v_min = in.v_min;
    ea.mo_ctx = in.motion ? in.mo_ctx : nullptr;
    const long long n_ctas = (long long)S * ea.ctas_per_scn;
    if (n_ctas > 0x7fffffffLL) return F1L_ERR_TOO_LARGE;
    if (!sp.empty) ec.fn()<<<(unsigned)n_ctas, ec.nw * 32, smem, stream>>>(ea);
    {
        const EvalBucket& b = *ec.bucket;
        const int info[11] = {b.ipl, b.s, b.sg, ec.nw, ec.build->minb, ea.chunk, ea.ctas_per_scn, ea.item,
                              (int)ec.persistent, (int)ec.pw, (int)ec.mo};
        for (int i = 0; i < 11; ++i) h->eval_info[i] = info[i];
    }
    if (time_it) cudaEventRecord(ev[2], stream);

    ec.bucket->select<<<S, SELECT_THREADS, 0, stream>>>(select_args(h, in, sc, o));
    if (time_it) {
        cudaEventRecord(ev[3], stream);
        h->timed = 1;
        h->ev_next = (h->ev_next + 1) % F1L_EV_SLOTS;
        if (h->ev_count < F1L_EV_SLOTS) h->ev_count++;
    }
    h->launches += 3;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, e, "pipeline launch");
    return F1L_OK;
}

// result block of a single query (h_out, mapped pinned memory that select_kernel writes): header
// then the best trajectory, everything a plain plan() call returns
struct QHeader {
    double steer, speed;                 // +0
    int32_t best_idx;                    // +16
    int32_t no_feasible, tracker_found;  // +20
    int32_t xchg_status;                 // +28 sharded query: != 0 when a peer did not arrive
    float best_cost;                     // +32
    float pad2[3];                       // -> 48 bytes, keeps the float4 trajectory 16-aligned
};
static_assert(sizeof(QHeader) == 48, "QHeader layout");
// result block: header | best trajectory float4[F1L_MAX_M] | map-frame trajectory double[F1L_MAX_M][4]
#define Q_OFF_TRAJ (sizeof(QHeader))
#define Q_OFF_MAP (Q_OFF_TRAJ + F1L_MAX_M * sizeof(float4))
#define Q_RES_BYTES (Q_OFF_MAP + F1L_MAX_M * 4 * sizeof(double))

// select_kernel's outputs of a single query: the result block as the device sees it
BatchOut q_result_out(f1l_handle h, bool want_map) {
    char* dres = (char*)h->h_out_dev;
    BatchOut o;
    o.steer_speed = (double*)(dres + offsetof(QHeader, steer));
    o.best_idx = (int32_t*)(dres + offsetof(QHeader, best_idx));
    o.status = (int32_t*)(dres + offsetof(QHeader, no_feasible));
    o.best_cost = (float*)(dres + offsetof(QHeader, best_cost));
    o.best_traj = (float4*)(dres + Q_OFF_TRAJ);
    o.best_traj_map = want_map ? (double*)(dres + Q_OFF_MAP) : nullptr;
    return o;
}

// the result block into the caller's f1l_plan_result (after the stream synchronise)
void q_copy_result(f1l_handle h, int C, f1l_plan_result* out) {
    const int M = h->cfg.n_samples;
    const char* res = (const char*)h->h_out.p;
    const QHeader* hd = (const QHeader*)res;
    out->steer = hd->steer;
    out->speed = hd->speed;
    out->best_idx = hd->best_idx;
    out->no_feasible = hd->no_feasible;
    out->tracker_found = hd->tracker_found;
    out->n_candidates = C;
    out->best_cost = hd->best_cost;
    if (out->best_traj) memcpy(out->best_traj, res + Q_OFF_TRAJ, (size_t)M * 16);
    if (out->best_traj_map) memcpy(out->best_traj_map, res + Q_OFF_MAP, (size_t)M * 32);
}

// pinned-host / device input block of a single query (fixed size, so that the copy is a constant
// node of the CUDA graph): the opponent count travels in the block, not as a kernel argument
struct QInput {
    double pose[4];
    int32_t n_opp, pad;
    double opp[3 * F1L_MAX_OPP];
    double opp_vel[2 * F1L_MAX_OPP];   // f1l_plan_motion
};
static_assert(sizeof(QInput) <= 1024, "QInput fits the pinned staging block");

// the checks every moving-opponent entry point makes on v_min and the velocity pointer
int check_motion(int n_opp, const double* opp_vel, double v_min) {
    if (!std::isfinite(v_min) || !(v_min > 0.0)) return F1L_ERR_INVALID_ARG;
    if (n_opp > 0 && !opp_vel) return F1L_ERR_INVALID_ARG;
    return F1L_OK;
}

}  // namespace

extern "C" {

int f1l_default_config(f1l_config* c) {
    if (!c) return F1L_ERR_INVALID_ARG;
    memset(c, 0, sizeof(*c));
    c->n_samples = 100;
    c->n_newton = 8;
    c->window = 128;
    c->n_shift = 5;
    c->n_cull = 10;
    c->literal_tracker = 0;
    c->use_goal_kappa = 0;
    c->weights[0] = 0.1;
    c->weights[1] = 0.1;
    c->weights[2] = 0.1;
    c->weights[3] = 0.2;
    c->weights[4] = 0.5;
    c->kappa_max = std::tan(0.4189) / 0.33;
    c->car_length = 0.58;
    c->car_width = 0.31;
    c->converge_tol = 1e-4;
    c->tracker_lookahead = 0.8;
    c->wheelbase = 0.33;
    c->max_reacquire = 20.0;
    return F1L_OK;
}

const char* f1l_strerror(int code) {
    switch (code) {
        case F1L_OK: return "ok";
        case F1L_ERR_INVALID_ARG: return "invalid argument";
        case F1L_ERR_NO_TRACK: return "no track uploaded (f1l_set_track)";
        case F1L_ERR_CUDA: return "CUDA error (see f1l_last_cuda_error)";
        case F1L_ERR_NO_DEVICE: return "no CUDA device / device index out of range";
        case F1L_ERR_TOO_LARGE: return "problem too large for this build (window / grid limits)";
        case F1L_ERR_NO_GOALS: return "no goal grid set (f1l_set_goal_grid) and no explicit goals";
        case F1L_ERR_ALLOC: return "host allocation failed";
        case F1L_ERR_PEER_TIMEOUT: return "a peer rank did not arrive at the sharded-query exchange";
        default: return "unknown f1l status";
    }
}

const char* f1l_last_cuda_error(f1l_handle h) { return h ? h->err : ""; }
int f1l_device(f1l_handle h) { return h ? h->device : -1; }
int64_t f1l_launch_count(f1l_handle h) { return h ? h->launches : 0; }

int f1l_get_stats(f1l_handle h, uint64_t* out, int n) {
    if (!h || !out || n < 2) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaDeviceSynchronize());   // batch pipelines run on their own streams
    unsigned long long v[2] = {0, 0};
    CK(cudaMemcpy(v, h->stats.p, sizeof(v), cudaMemcpyDeviceToHost));
    CK(cudaMemset(h->stats.p, 0, sizeof(v)));
    out[0] = v[0];
    out[1] = v[1];
    return F1L_OK;
}

int f1l_set_stats(f1l_handle h, int on) {
    if (!h) return F1L_ERR_INVALID_ARG;
    h->stats_on = on != 0;
    h->epoch++;   // a kernel argument of the captured graph
    return F1L_OK;
}

int f1l_debug_eval_plan(int n_cand, int n_scenarios, int M, int sm_count, int generator,
                        int32_t* out, int n) {
    return f1l_debug_eval_choice(n_cand, n_scenarios, M, sm_count, generator, 0, out, n < 4 ? n : 4);
}

int f1l_debug_eval_choice(int n_cand, int n_scenarios, int M, int sm_count, int generator, int flags,
                          int32_t* out, int n) {
    if (!out || n < 4 || n_cand <= 0 || n_scenarios <= 0 || M < 2 || M > F1L_MAX_M || sm_count <= 0 ||
        (flags & ~(F1L_EVAL_LONE | F1L_EVAL_WEIGHTS)) || ((flags & F1L_EVAL_LONE) && n_scenarios != 1))
        return F1L_ERR_INVALID_ARG;
    const EvalChoice c = choose_eval(n_cand, n_scenarios, M, sm_count, generator == 0,
                                     (flags & F1L_EVAL_LONE) != 0, (flags & F1L_EVAL_WEIGHTS) != 0);
    const EvalBucket& b = *c.bucket;
    // minb 0: the choice names an instance that is not built (launch_pipeline refuses it)
    const int v[13] = {c.nw, c.chunk, c.ctas_per_scn, c.item, b.m_max, b.ipl, b.s, b.sg,
                       c.fn() ? c.build->minb : 0, (int)c.wide, (int)c.persistent, (int)c.pw,
                       ((EVAL_SMEM_MAX - (int)c.build->smem_fixed) / 32 - EVAL_SEG_PAD) & ~31};
    for (int i = 0; i < n && i < 13; ++i) out[i] = v[i];
    return F1L_OK;
}

int f1l_debug_eval_builds(int32_t* out, int n) {
    const int rows = (int)(sizeof(kEvalBuckets) / sizeof(kEvalBuckets[0]));
    if (!out || n < 8 * rows) return F1L_ERR_INVALID_ARG;
    for (int r = 0; r < rows; ++r) {
        const EvalBucket& b = kEvalBuckets[r];
        const int v[8] = {b.m_max, b.ipl, b.s, b.sg, b.nw4.minb, b.nw7.minb, b.nw8.minb, b.wide.minb};
        for (int i = 0; i < 8; ++i) out[8 * r + i] = v[i];
    }
    return rows;
}

int f1l_debug_pp_parts(int n_poses, int n_waypoints, int slots) {
    if (n_poses <= 0 || n_waypoints < 2 || slots <= 0) return F1L_ERR_INVALID_ARG;
    return pp_task_parts((n_poses + PP_CTA_POSES - 1) / PP_CTA_POSES, (n_waypoints - 1 + 31) >> 5, slots);
}

int f1l_last_eval_shape(f1l_handle h, int32_t* out, int n) {
    if (!h || !out || n < 8) return F1L_ERR_INVALID_ARG;
    for (int i = 0; i < n && i < 11; ++i) out[i] = h->eval_info[i];
    return F1L_OK;
}

int f1l_set_graph(f1l_handle h, int on) {
    if (!h) return F1L_ERR_INVALID_ARG;
    h->use_graph = on;
    return F1L_OK;
}

int f1l_set_timing(f1l_handle h, int on) {
    if (!h) return F1L_ERR_INVALID_ARG;
    h->timing = on;
    h->ev_next = 0;
    h->ev_count = 0;
    h->timed = 0;
    return F1L_OK;
}

int f1l_last_kernel_ms(f1l_handle h, float* sample_ms, float* eval_ms, float* select_ms) {
    if (!h) return F1L_ERR_INVALID_ARG;
    if (h->timing && h->timed) {
        CK(cudaSetDevice(h->device));
        cudaEvent_t* ev = h->ev + 4 * ((h->ev_next + F1L_EV_SLOTS - 1) % F1L_EV_SLOTS);
        CK(cudaEventSynchronize(ev[3]));
        cudaEventElapsedTime(&h->last_ms[0], ev[0], ev[1]);
        cudaEventElapsedTime(&h->last_ms[1], ev[1], ev[2]);
        cudaEventElapsedTime(&h->last_ms[2], ev[2], ev[3]);
    }
    if (sample_ms) *sample_ms = h->last_ms[0];
    if (eval_ms) *eval_ms = h->last_ms[1];
    if (select_ms) *select_ms = h->last_ms[2];
    return F1L_OK;
}

int f1l_mean_kernel_ms(f1l_handle h, float* sample_ms, float* eval_ms, float* select_ms,
                       int* n_launches) {
    if (!h) return F1L_ERR_INVALID_ARG;
    double acc[3] = {0, 0, 0};
    const int n = h->ev_count;
    if (n > 0) {
        CK(cudaSetDevice(h->device));
        for (int k = 0; k < n; ++k) {
            cudaEvent_t* ev = h->ev + 4 * ((h->ev_next + F1L_EV_SLOTS - 1 - k) % F1L_EV_SLOTS);
            CK(cudaEventSynchronize(ev[3]));
            for (int j = 0; j < 3; ++j) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, ev[j], ev[j + 1]);
                acc[j] += ms;
            }
        }
    }
    if (sample_ms) *sample_ms = n ? (float)(acc[0] / n) : 0.f;
    if (eval_ms) *eval_ms = n ? (float)(acc[1] / n) : 0.f;
    if (select_ms) *select_ms = n ? (float)(acc[2] / n) : 0.f;
    if (n_launches) *n_launches = n;
    return F1L_OK;
}

int f1l_set_config(f1l_handle h, const f1l_config* cfg) {
    if (!h) return F1L_ERR_INVALID_ARG;
    int r = check_config(cfg);
    if (r != F1L_OK) return r;
    if (cfg->n_samples != h->cfg.n_samples) h->has_prev = 0;
    h->cfg = *cfg;
    h->epoch++;
    return F1L_OK;
}

int f1l_get_config(f1l_handle h, f1l_config* cfg) {
    if (!h || !cfg) return F1L_ERR_INVALID_ARG;
    *cfg = h->cfg;
    return F1L_OK;
}

static int build_lut(f1l_handle h) {
    const int cells = h->ldims[0] * h->ldims[1] * h->ldims[2];
    ENS(h->lut, (size_t)cells * sizeof(float4));
    lut_build_kernel<<<(cells + 127) / 128, 128, 0, h->stream>>>(
        (float4*)h->lut.p, h->ldims[0], h->ldims[1], h->ldims[2], h->lranges[0], h->lranges[1],
        h->lranges[2], h->lranges[3], h->lranges[4], h->lranges[5]);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return F1L_OK;
}

int f1l_create(f1l_handle* out, int device, const f1l_config* cfg) {
    if (!out) return F1L_ERR_INVALID_ARG;
    *out = nullptr;
    f1l_config c;
    if (cfg) c = *cfg;
    else f1l_default_config(&c);
    int r = check_config(&c);
    if (r != F1L_OK) return r;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count)
        return F1L_ERR_NO_DEVICE;
    f1l_handle h = new (std::nothrow) f1l_ctx();
    if (!h) return F1L_ERR_ALLOC;
    h->device = device;
    h->cfg = c;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 4 * F1L_EV_SLOTS && e == cudaSuccess; ++i) e = cudaEventCreate(&h->ev[i]);
    for (int i = 0; i < N_PIPE && e == cudaSuccess; ++i)
        e = cudaStreamCreateWithFlags(&h->pipe[i].stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaHostAlloc(&h->h_in.p, 1024, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaHostAlloc(&h->h_out.p, Q_RES_BYTES, cudaHostAllocMapped);
    // single queries write their results straight into h_out: no mapping, no handle
    if (e == cudaSuccess) e = cudaHostGetDevicePointer(&h->h_out_dev, h->h_out.p, 0);
    if (e == cudaSuccess) {
        memset(h->h_in.p, 0, 1024);
        memset(h->h_out.p, 0, Q_RES_BYTES);
    }
    if (e == cudaSuccess) {
        int sm = 0;
        cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
        if (sm > 0) h->sm_count = sm;
        // opt in to large dynamic shared memory for every eval instantiation
        for (const EvalBucket& b : kEvalBuckets) {
            for (const EvalBuild* eb : {&b.nw4, &b.nw7, &b.nw8, &b.wide}) {
                for (eval_fn fn : {eb->fn, eb->fn_w, eb->fn_m}) {
                    if (!fn) continue;
                    cudaError_t e2 = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, EVAL_SMEM_MAX);
                    if (e2 != cudaSuccess && e == cudaSuccess) e = e2;
                }
            }
        }
    }
    if (e != cudaSuccess) {
        fail(h, e, "f1l_create");
        f1l_destroy(h);
        return F1L_ERR_CUDA;
    }
    r = build_lut(h);
    if (r == F1L_OK) r = ensure(h, h->stats, 2 * sizeof(unsigned long long));
    if (r == F1L_OK && cudaMemsetAsync(h->stats.p, 0, 2 * sizeof(unsigned long long), h->stream) != cudaSuccess)
        r = F1L_ERR_CUDA;
    if (r != F1L_OK) {
        f1l_destroy(h);
        return r;
    }
    *out = h;
    return F1L_OK;
}

int f1l_destroy(f1l_handle h) {
    if (!h) return F1L_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    f1l_xchg_detach(h);
    for (int i = 0; i < N_PIPE; ++i)
        if (h->pipe[i].stream) cudaStreamDestroy(h->pipe[i].stream);
    if (h->gexec) cudaGraphExecDestroy(h->gexec);
    for (int i = 0; i < 4 * F1L_EV_SLOTS; ++i)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;   // frees every device and pinned buffer
    return F1L_OK;
}

int f1l_set_track(f1l_handle h, const double* wpts, int n, int ncols) {
    if (!h || !wpts || n < 2 || ncols < 2) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    const int nseg = n - 1;
    const int nblk = (nseg + 31) / 32;
    std::vector<double> xy(2 * (size_t)n), v(n, 0.0), psi(n, 0.0), kap(n, 0.0);
    for (int i = 0; i < n; ++i) {
        xy[2 * i] = wpts[(size_t)i * ncols];
        xy[2 * i + 1] = wpts[(size_t)i * ncols + 1];
        if (ncols > 2) v[i] = wpts[(size_t)i * ncols + 2];
        if (ncols > 3) psi[i] = wpts[(size_t)i * ncols + 3];
        if (ncols > 4) kap[i] = wpts[(size_t)i * ncols + 4];
    }
    std::vector<float> segA(4 * (size_t)nseg), segB(2 * (size_t)nseg);
    std::vector<double> blk(2 * (size_t)nblk), seg_s(2 * (size_t)nseg);
    for (int b = 0; b < nblk; ++b) {
        blk[2 * b] = xy[2 * (size_t)(32 * b)];
        blk[2 * b + 1] = xy[2 * (size_t)(32 * b) + 1];
    }
    for (int k = 0; k < nseg; ++k) {
        const double ox = blk[2 * (k / 32)], oy = blk[2 * (k / 32) + 1];
        const double ax = xy[2 * k] - ox, ay = xy[2 * k + 1] - oy;
        const double dx = xy[2 * k + 2] - xy[2 * k], dy = xy[2 * k + 3] - xy[2 * k + 1];
        const double len = std::sqrt(dx * dx + dy * dy);
        seg_s[2 * k] = k ? seg_s[2 * k - 2] + seg_s[2 * k - 1] : 0.0;
        seg_s[2 * k + 1] = len;
        const double ux = dx / len, uy = dy / len;
        const double sc = (double)TRACK_SCALE, hh = 0.5 * len;   // table units (track_seg_d2)
        segA[4 * k] = (float)ux;
        segA[4 * k + 1] = (float)uy;
        segA[4 * k + 2] = (float)(-(ax * ux + ay * uy + hh) * sc);
        segA[4 * k + 3] = (float)(-(-ax * uy + ay * ux) * sc);
        segB[2 * k] = (float)(-hh * sc);
        segB[2 * k + 1] = (float)(-uy);
    }
    ENS(h->xy, xy.size() * 8);
    ENS(h->v, v.size() * 8);
    ENS(h->psi, psi.size() * 8);
    ENS(h->kappa, kap.size() * 8);
    ENS(h->segA, segA.size() * 4);
    ENS(h->segB, segB.size() * 4);
    ENS(h->blk, blk.size() * 8);
    ENS(h->seg_s, seg_s.size() * 8);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->xy.p, xy.data(), xy.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->v.p, v.data(), v.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->psi.p, psi.data(), psi.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->kappa.p, kap.data(), kap.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->segA.p, segA.data(), segA.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->segB.p, segB.data(), segB.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->blk.p, blk.data(), blk.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->seg_s.p, seg_s.data(), seg_s.size() * 8, cudaMemcpyHostToDevice));
    {
        const double gx = xy[0] - xy[2 * (size_t)nseg], gy = xy[1] - xy[2 * (size_t)nseg + 1];
        h->lap = seg_s[2 * (size_t)nseg - 2] + seg_s[2 * (size_t)nseg - 1] + std::sqrt(gx * gx + gy * gy);
    }
    // the scan's constant-memory copy: one table per device, taken over by the latest upload (no
    // kernel of another handle may still be reading it: device-wide sync, this is the slow path)
    h->ctab_key = 0;
    if (nblk * 32 <= F1L_CTAB_SEGS && h->device >= 0 && h->device < 64) {
        {   // withdraw the table from whoever owns it, then wait for the scans already enqueued on it
            std::lock_guard<std::mutex> lk(g_ctab_mu);
            g_ctab_owner[h->device] = 0;
        }
        CK(cudaDeviceSynchronize());
        // padded to whole 32-segment blocks with entries no query point comes near (d^2 = 1e18 table
        // units): the constant-memory scan has no partial-block path
        std::vector<float> cA(segA), cB(segB);
        for (int k = nseg; k < nblk * 32; ++k) {
            const float far_a[4] = {1.0f, 0.0f, -1e9f, -1e9f}, far_b[2] = {-1.0f, -0.0f};
            cA.insert(cA.end(), far_a, far_a + 4);
            cB.insert(cB.end(), far_b, far_b + 2);
        }
        CK(cudaMemcpyToSymbol(c_segA, cA.data(), cA.size() * 4));
        CK(cudaMemcpyToSymbol(c_segB, cB.data(), cB.size() * 4));
        {
            std::lock_guard<std::mutex> lk(g_ctab_mu);
            h->ctab_key = ++g_ctab_serial;
            g_ctab_owner[h->device] = h->ctab_key;
        }
    }
    h->epoch++;
    h->n = n;
    h->ncols = ncols;
    return F1L_OK;
}

int f1l_set_grid(f1l_handle h, const uint8_t* occ, int height, int width, double ox, double oy,
                 double res) {
    if (!h || !occ || height <= 0 || width <= 0 || !(res > 0)) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    ENS(h->grid, (size_t)height * width);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->grid.p, occ, (size_t)height * width, cudaMemcpyHostToDevice));
    ENS(h->clear, (size_t)height * width * sizeof(uint16_t));
    ENS(h->clear_tmp, (size_t)height * width);
    ENS(h->edt, (size_t)height * width * sizeof(uint16_t));
    {
        dim3 blk(256), grd((width + 255) / 256, height);
        clearance_h_kernel<<<grd, blk, 0, h->stream>>>((const uint8_t*)h->grid.p, height, width,
                                                       (uint8_t*)h->clear_tmp.p);
        clearance_v_kernel<<<grd, blk, 0, h->stream>>>((const uint8_t*)h->clear_tmp.p, height, width,
                                                       (uint16_t*)h->clear.p);
        edt_v_kernel<<<grd, blk, 0, h->stream>>>((const uint8_t*)h->clear_tmp.p, height, width,
                                                 (uint16_t*)h->edt.p);
        h->launches += 3;
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(h->stream));
    }
    h->gh = height;
    h->gw = width;
    h->gox = ox;
    h->goy = oy;
    h->epoch++;
    h->gres = res;
    return F1L_OK;
}

int f1l_clear_grid(f1l_handle h) {
    if (!h) return F1L_ERR_INVALID_ARG;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    h->grid.reset();
    h->clear.reset();
    h->clear_tmp.reset();
    h->edt.reset();
    h->epoch++;
    h->gh = h->gw = 0;
    return F1L_OK;
}

int f1l_get_edt(f1l_handle h, uint16_t* out) {
    if (!h || !out || !h->edt.p || h->gh <= 0) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out, h->edt.p, (size_t)h->gh * h->gw * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    return F1L_OK;
}

int f1l_set_goal_grid(f1l_handle h, const double* lookaheads, int nL, const double* widths,
                      int nW) {
    if (!h || !lookaheads || !widths || nL <= 0 || nW <= 0 || nL > F1L_MAX_LOOKAHEADS)
        return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    std::vector<float> wf(nW);
    for (int i = 0; i < nW; ++i) wf[i] = (float)widths[i];
    ENS(h->lookaheads, (size_t)nL * 8);
    ENS(h->widths, (size_t)nW * 4);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->lookaheads.p, lookaheads, (size_t)nL * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->widths.p, wf.data(), (size_t)nW * 4, cudaMemcpyHostToDevice));
    h->epoch++;
    h->nL = nL;
    h->nW = nW;
    return F1L_OK;
}

int f1l_get_lut_shape(f1l_handle h, int32_t dims[3], double ranges[6]) {
    if (!h) return F1L_ERR_INVALID_ARG;
    for (int i = 0; i < 3; ++i) dims[i] = h->ldims[i];
    for (int i = 0; i < 6; ++i) ranges[i] = h->lranges[i];
    return F1L_OK;
}

int f1l_get_lut(f1l_handle h, float* out) {
    if (!h || !out) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out, h->lut.p, (size_t)h->ldims[0] * h->ldims[1] * h->ldims[2] * sizeof(float4),
                  cudaMemcpyDeviceToHost));
    return F1L_OK;
}

int f1l_set_lut(f1l_handle h, const float* lut, const int32_t dims[3], const double ranges[6]) {
    if (!h || !lut || !dims || !ranges) return F1L_ERR_INVALID_ARG;
    if (dims[0] <= 0 || dims[1] <= 0 || dims[2] <= 0) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    const size_t bytes = (size_t)dims[0] * dims[1] * dims[2] * sizeof(float4);
    ENS(h->lut, bytes);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->lut.p, lut, bytes, cudaMemcpyHostToDevice));
    for (int i = 0; i < 3; ++i) h->ldims[i] = dims[i];
    h->epoch++;
    for (int i = 0; i < 6; ++i) h->lranges[i] = ranges[i];
    return F1L_OK;
}

int f1l_set_prev_path(f1l_handle h, const float* theta_prev, int m) {
    if (!h || !theta_prev || m != h->cfg.n_samples) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    ENS(h->prev, F1L_MAX_M * sizeof(float));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->prev.p, theta_prev, (size_t)m * sizeof(float), cudaMemcpyHostToDevice));
    h->has_prev = 1;
    h->prev_m = m;
    return F1L_OK;
}

int f1l_clear_prev_path(f1l_handle h) {
    if (!h) return F1L_ERR_INVALID_ARG;
    h->has_prev = 0;
    return F1L_OK;
}

// ---- single query -------------------------------------------------------------------------
// opp_vel / v_min: moving opponents (f1l_plan_motion; motion false: static)
static int plan_internal(f1l_handle h, const double pose[4], const double* opp, int n_opp,
                         const double* goals, int n_goals, const Shard& shard, bool exchange,
                         int update_prev, f1l_plan_result* out, bool motion = false,
                         const double* opp_vel = nullptr, double v_min = 1.0) {
    if (!h || !pose || !out) return F1L_ERR_INVALID_ARG;
    if (n_opp < 0 || n_opp > F1L_MAX_OPP || (n_opp > 0 && !opp)) return F1L_ERR_INVALID_ARG;
    if (motion) {
        if (const int r = check_motion(n_opp, opp_vel, v_min); r != F1L_OK) return r;
        for (int k = 0; k < 2 * n_opp; ++k)
            if (!std::isfinite(opp_vel[k])) return F1L_ERR_INVALID_ARG;
    }
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    CK(cudaSetDevice(h->device));
    exchange = exchange && h->xview.world > 1;
    PipeIn in;
    if (const int r = make_span(h, n_goals, shard, exchange, in.span); r != F1L_OK) return r;
    const Span& sp = in.span;
    const int C = sp.C, M = h->cfg.n_samples;
    cudaStream_t st = h->stream;

    NvtxRange nvtx_plan("f1l.plan (single query)");
    // stage inputs (pinned)
    QInput* hin = (QInput*)h->h_in.p;
    memcpy(hin->pose, pose, 4 * sizeof(double));
    hin->n_opp = n_opp;
    hin->pad = 0;
    if (n_opp) memcpy(hin->opp, opp, (size_t)n_opp * 3 * sizeof(double));
    if (motion && n_opp) memcpy(hin->opp_vel, opp_vel, (size_t)n_opp * 2 * sizeof(double));
    ENS(h->q_in, sizeof(QInput));
    if (motion) ENS(h->mo_dbg, (1 + 2 * F1L_MAX_OPP) * sizeof(float));
    if (const int r = h->q_scratch.reserve(h, 1); r != F1L_OK) return r;
    ENS(h->prev, F1L_MAX_M * sizeof(float));
    // detail block layout (every region 16-byte aligned)
    const size_t c16 = ((size_t)C + 3) & ~(size_t)3;
    const size_t off_costs = 0, off_terms = off_costs + c16 * 4, off_goals = off_terms + c16 * F1L_N_TERMS * 4;
    const size_t off_params = off_goals + c16 * 12, off_flags = off_params + c16 * 16;
    const size_t detail_bytes = off_flags + c16;
    ENS(h->q_detail, detail_bytes);
    const bool want_detail = out->costs || out->terms || out->flags || out->goals || out->params;
    if (want_detail && h->h_detail.cap < detail_bytes) {
        CK(cudaStreamSynchronize(st));
        h->h_detail.reset();
        CK(cudaHostAlloc(&h->h_detail.p, detail_bytes, cudaHostAllocDefault));
        h->h_detail.cap = detail_bytes;
        h->epoch++;   // the captured graph holds the old staging address
    }
    char* ddet = (char*)h->q_detail.p;
    // the big optional arrays go straight into the caller's buffers
    const Stage big[] = {{&h->q_states, nullptr, out->states, (size_t)M * 16},
                         {&h->q_headings, nullptr, out->headings, (size_t)M * 8}};
    if (const int r = stage_in(h, st, big, 0, C); r != F1L_OK) return r;
    std::vector<float> g4;
    if (goals) {
        if (const int r = upload_goals(h, goals, C, g4, st); r != F1L_OK) return r;
        CK(cudaStreamSynchronize(st));  // g4 is a stack-lifetime staging buffer
        in.goals = (const float4*)h->q_goals.p;
    }

    // Results of a single query: the select kernel writes header and best trajectory straight into
    // the mapped pinned block (posted writes over the host link, 3-10 KB) -- no D2H copy node on the
    // latency path.
    BatchOut o = q_result_out(h, out->best_traj_map != nullptr);
    o.costs = (float*)(ddet + off_costs);
    o.terms = out->terms ? (float*)(ddet + off_terms) : nullptr;
    o.flags = out->flags ? (uint8_t*)(ddet + off_flags) : nullptr;
    o.goals_out = out->goals ? (float*)(ddet + off_goals) : nullptr;
    o.params = out->params ? (float4*)(ddet + off_params) : nullptr;
    o.states = (float4*)big[0].dev();
    o.headings = (float2*)big[1].dev();
    o.prev_out = update_prev ? (float*)h->prev.p : nullptr;
    if (exchange) {   // the ranks' minima meet inside select_kernel (peer memory over NVLink)
        in.xc = &h->xview;
        o.xchg_status = (int32_t*)((char*)h->h_out_dev + offsetof(QHeader, xchg_status));
    }
    const bool sharded = exchange || sp.row_step > 1 || sp.c_begin > 0 || sp.c_end < C;
    const QInput* din = (const QInput*)h->q_in.p;
    in.poses = din->pose;
    in.opp = din->opp;
    in.n_opp = &din->n_opp;
    in.S = 1;
    in.max_opp = F1L_MAX_OPP;
    in.prev_theta = h->has_prev ? (const float*)h->prev.p : nullptr;
    in.work_next = (int*)((char*)h->q_scratch.best.p + 8);   // behind the one argmin key
    if (motion) {
        in.motion = true;
        in.opp_vel = din->opp_vel;
        in.v_min = v_min;
        in.mo_ctx = (float*)h->mo_dbg.p;
    }
    // H2D of the input block, the three kernels, D2H of the detail block.  The similarity term
    // reads the previous path while select overwrites it: eval reads it before select runs
    // (stream order), so one buffer suffices.
    auto enqueue = [&](bool time_it) -> int {
        CK(cudaMemcpyAsync(h->q_in.p, hin, sizeof(QInput), cudaMemcpyHostToDevice, st));
        if (sharded && want_detail) {
            // sharded evaluation: untouched candidates keep +inf / zero flags (only when the
            // per-candidate arrays travel back at all)
            fill_f32_kernel<<<(C + 255) / 256, 256, 0, st>>>(o.costs, (size_t)C, INFINITY);
            h->launches += 1;
            if (o.flags) CK(cudaMemsetAsync(o.flags, 0, (size_t)C, st));
        }
        int r = launch_pipeline(h, st, in, h->q_scratch, o, time_it);
        if (r != F1L_OK) return r;
        if (want_detail)
            CK(cudaMemcpyAsync(h->h_detail.p, ddet, detail_bytes, cudaMemcpyDeviceToHost, st));
        return F1L_OK;
    };
    if (h->use_graph && !goals && !h->timing) {
        // the whole chain as one CUDA graph, re-captured only when an upload / config change, the
        // set of requested outputs or the span (a constant of the captured kernels too) alters a
        // kernel argument
        const unsigned long long mask = (want_detail ? 256u : 0u) | (out->terms ? 1u : 0u) | (out->flags ? 2u : 0u) |
                                        (out->goals ? 4u : 0u) | (out->params ? 8u : 0u) |
                                        (out->states ? 16u : 0u) | (out->headings ? 32u : 0u) |
                                        (update_prev ? 64u : 0u) | (h->has_prev ? 128u : 0u) |
                                        (exchange ? 512u : 0u) | (out->best_traj_map ? 1024u : 0u) |
                                        (motion ? 2048u : 0u);
        if (!h->gexec || h->gkey[0] != h->epoch || h->gkey[1] != mask || memcmp(&h->gspan, &sp, sizeof(Span)) ||
            (motion && h->gvmin != v_min)) {
            if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; }
            const int64_t launches0 = h->launches;
            cudaGraph_t graph = nullptr;
            CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            int r = enqueue(false);
            cudaError_t ce = cudaStreamEndCapture(st, &graph);
            h->launches = launches0;
            if (r != F1L_OK) { if (graph) cudaGraphDestroy(graph); return r; }
            if (ce != cudaSuccess) return fail(h, ce, "cudaStreamEndCapture");
            ce = cudaGraphInstantiate(&h->gexec, graph, 0);
            cudaGraphDestroy(graph);
            if (ce != cudaSuccess) { h->gexec = nullptr; return fail(h, ce, "cudaGraphInstantiate"); }
            h->gkey[0] = h->epoch;
            h->gkey[1] = mask;
            h->gspan = sp;
            h->gvmin = motion ? v_min : 0.0;
        }
        CK(cudaGraphLaunch(h->gexec, st));
        h->launches += 3;
    } else {
        int r = enqueue(h->timing != 0);
        if (r != F1L_OK) return r;
    }

    if (const int r = stage_out(h, st, big, 0, C); r != F1L_OK) return r;
    CK(cudaStreamSynchronize(st));
    if (update_prev) {
        h->has_prev = 1;
        h->prev_m = M;
    }
    if (exchange && ((const QHeader*)h->h_out.p)->xchg_status != 0) return F1L_ERR_PEER_TIMEOUT;
    h->lastq_span = sp;
    h->lastq_goals = goals != nullptr;
    h->lastq_epoch = h->epoch;
    q_copy_result(h, C, out);
    if (want_detail) {
        const char* hdet = (const char*)h->h_detail.p;
        if (out->costs) memcpy(out->costs, hdet + off_costs, (size_t)C * 4);
        if (out->terms) memcpy(out->terms, hdet + off_terms, (size_t)C * F1L_N_TERMS * 4);
        if (out->flags) memcpy(out->flags, hdet + off_flags, (size_t)C);
        if (out->goals) memcpy(out->goals, hdet + off_goals, (size_t)C * 12);
        if (out->params) memcpy(out->params, hdet + off_params, (size_t)C * 16);
    }
    return F1L_OK;
}

int f1l_plan(f1l_handle h, const double pose[4], const double* opp, int n_opp, int update_prev,
             f1l_plan_result* out) {
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, Shard{}, false, update_prev, out);
}

int f1l_plan_motion(f1l_handle h, const double pose[4], const double* opp, const double* opp_vel, int n_opp,
                    double v_min, int update_prev, f1l_plan_result* out) {
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, Shard{}, false, update_prev, out, true, opp_vel, v_min);
}

int f1l_debug_motion_ctx(f1l_handle h, float* out, int n) {
    if (!h || !out || n < 1 + 2 * F1L_MAX_OPP || !h->mo_dbg.p) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out, h->mo_dbg.p, (1 + 2 * F1L_MAX_OPP) * sizeof(float), cudaMemcpyDeviceToHost));
    return F1L_OK;
}

int f1l_plan_shard(f1l_handle h, const double pose[4], const double* opp, int n_opp, int c_begin,
                   int c_end, f1l_plan_result* out) {
    // with peers attached (f1l_xchg_attach) every rank returns the GLOBAL winner
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, Shard{c_begin, c_end, 0, 1}, true, 0, out);
}

int f1l_plan_rows(f1l_handle h, const double pose[4], const double* opp, int n_opp, int row_begin,
                  int row_step, int update_prev, f1l_plan_result* out) {
    if (row_step < 1) return F1L_ERR_INVALID_ARG;
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, Shard{0, 0, row_begin, row_step}, true,
                         update_prev, out);
}

int f1l_select_candidate(f1l_handle h, int idx, float cost, int update_prev, f1l_plan_result* out) {
    if (!h || !out) return F1L_ERR_INVALID_ARG;
    // the sampler context, goal centres / explicit goals of the last query must still be current
    if (h->lastq_epoch != h->epoch || idx < 0 || idx >= h->lastq_span.C) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int M = h->cfg.n_samples;
    unsigned long long* hkey = (unsigned long long*)h->h_in.p;   // pinned staging
    uint32_t cb;
    memcpy(&cb, &cost, 4);
    const uint32_t ord = (cb & 0x80000000u) ? ~cb : (cb | 0x80000000u);   // float_orderable
    *hkey = ((unsigned long long)ord << 32) | (unsigned)idx;
    CK(cudaMemcpyAsync(h->q_scratch.best.p, hkey, 8, cudaMemcpyHostToDevice, st));
    PipeIn in;
    in.S = 1;
    in.goals = h->lastq_goals ? (const float4*)h->q_goals.p : nullptr;
    in.span = h->lastq_span;
    BatchOut o = q_result_out(h, out->best_traj_map != nullptr);
    o.prev_out = update_prev ? (float*)h->prev.p : nullptr;
    eval_bucket_of(M).select<<<1, SELECT_THREADS, 0, st>>>(select_args(h, in, h->q_scratch, o));
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    if (update_prev) { h->has_prev = 1; h->prev_m = M; }
    q_copy_result(h, in.span.C, out);
    return F1L_OK;
}

// ---- peer-memory exchange (CUDA IPC over NVLink P2P) -----------------------------------------
int f1l_xchg_export(f1l_handle h, uint8_t* handle_out, int n) {
    if (!h || !handle_out || n < (int)sizeof(cudaIpcMemHandle_t)) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (h->xview.world > 1) return F1L_ERR_INVALID_ARG;   // detach first
    // a whole 2 MB allocation granule of its own: the IPC handle maps exactly this block
    ENS(h->xchg, (size_t)2 << 20);
    unsigned long long init[F1L_XCHG_WORDS];
    for (int i = 0; i < F1L_XCHG_WORDS; ++i) init[i] = 0ull;
    CK(cudaMemcpy(h->xchg.p, init, sizeof(init), cudaMemcpyHostToDevice));
    cudaIpcMemHandle_t mh;
    CK(cudaIpcGetMemHandle(&mh, h->xchg.p));
    memcpy(handle_out, &mh, sizeof(mh));
    return F1L_OK;
}

int f1l_xchg_attach(f1l_handle h, int rank, int world, const uint8_t* handles) {
    if (!h || !handles || world < 1 || world > F1L_MAX_RANKS || rank < 0 || rank >= world)
        return F1L_ERR_INVALID_ARG;
    if (!h->xchg.p || h->xview.world > 1) return F1L_ERR_INVALID_ARG;   // export first / detach first
    CK(cudaSetDevice(h->device));
    XchgView v;
    v.world = world;
    v.rank = rank;
    for (int r = 0; r < F1L_MAX_RANKS; ++r) v.peer[r] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (r == rank) { v.peer[r] = (unsigned long long*)h->xchg.p; continue; }
        cudaIpcMemHandle_t mh;
        memcpy(&mh, handles + (size_t)r * sizeof(mh), sizeof(mh));
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int q = 0; q < r; ++q)
                if (q != rank && v.peer[q]) cudaIpcCloseMemHandle(v.peer[q]);
            return fail(h, e, "cudaIpcOpenMemHandle");
        }
        v.peer[r] = (unsigned long long*)p;
    }
    h->xview = v;
    h->epoch++;   // a captured graph holds the old kernel arguments
    return F1L_OK;
}

int f1l_xchg_detach(f1l_handle h) {
    if (!h) return F1L_ERR_INVALID_ARG;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (int r = 0; r < h->xview.world; ++r)
        if (r != h->xview.rank && h->xview.peer[r]) cudaIpcCloseMemHandle(h->xview.peer[r]);
    h->xview.world = 0;
    h->xview.rank = 0;
    for (int r = 0; r < F1L_MAX_RANKS; ++r) h->xview.peer[r] = nullptr;
    h->epoch++;
    return F1L_OK;
}

int f1l_plan_goals(f1l_handle h, const double pose[4], const double* goals, int n_goals,
                   const double* opp, int n_opp, int update_prev, f1l_plan_result* out) {
    if (!goals || n_goals <= 0) return F1L_ERR_INVALID_ARG;
    return plan_internal(h, pose, opp, n_opp, goals, n_goals, Shard{}, false, update_prev, out);
}

int f1l_generate(f1l_handle h, const double* goals, int n_goals, float* states, float* params,
                 uint8_t* flags) {
    if (!h || !goals || n_goals <= 0 || !states) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    const int C = n_goals, M = h->cfg.n_samples;
    cudaStream_t st = h->stream;
    const Stage t[] = {{&h->q_states, nullptr, states, (size_t)M * 16},
                       {&h->q_params, nullptr, params, 16},
                       {&h->q_flags, nullptr, flags, 1}};
    if (const int r = stage_in(h, st, t, 0, C); r != F1L_OK) return r;
    std::vector<float> g4;   // outlives the copy: the call ends in a synchronise
    if (const int r = upload_goals(h, goals, C, g4, st); r != F1L_OK) return r;
    const int wpc = 8;
    eval_bucket_of(M).generate<<<(C + wpc - 1) / wpc, wpc * 32, 0, st>>>(
        lut_view(h), eval_params(h), (const float4*)h->q_goals.p, C, (float4*)t[0].dev(),
        (float4*)t[1].dev(), (uint8_t*)t[2].dev());
    h->launches += 1;
    CK(cudaGetLastError());
    if (const int r = stage_out(h, st, t, 0, C); r != F1L_OK) return r;
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

// ---- batch --------------------------------------------------------------------------------
// prev_theta [S,M] / has_prev [S] (nullable): per-scenario previous paths.  With update_prev the
// select kernel overwrites them in place with each scenario's best trajectory.  That is safe:
// eval_kernel reads a scenario's path in its prologue, and select_kernel writes it in a later
// kernel on the same stream.
// The arguments of a batch call over the whole goal grid, checked; device or host pointers alike
static int batch_args(f1l_handle h, const f1l_batch_call* b, PipeIn& in, BatchOut& o) {
    if (!h || !b || !b->poses || b->n_scenarios <= 0) return F1L_ERR_INVALID_ARG;
    if (b->max_opp < 0 || b->max_opp > F1L_MAX_OPP || (b->max_opp > 0 && !b->opp)) return F1L_ERR_INVALID_ARG;
    if ((b->update_prev || b->has_prev) && !b->prev_theta) return F1L_ERR_INVALID_ARG;
    if (const int r = make_span(h, 0, Shard{}, false, in.span); r != F1L_OK) return r;
    in.poses = b->poses;
    in.opp = b->max_opp > 0 ? b->opp : nullptr;
    in.n_opp = b->n_opp;
    in.S = b->n_scenarios;
    in.max_opp = b->max_opp;
    in.prev_theta = b->prev_theta;
    in.prev_stride = h->cfg.n_samples;
    in.prev_valid = b->has_prev;
    in.weights = b->weights;
    o.best_idx = b->best_idx;
    o.best_cost = b->best_cost;
    o.best_traj = (float4*)b->best_traj;
    o.costs = b->costs;
    o.terms = b->terms;
    o.flags = b->flags;
    o.steer_speed = b->steer_speed;
    o.prev_out = b->update_prev ? b->prev_theta : nullptr;
    o.prev_valid_out = b->update_prev ? b->has_prev : nullptr;
    return F1L_OK;
}

static int plan_batch_dev_internal(f1l_handle h, const PipeIn& in, const BatchOut& o, cudaStream_t stream) {
    CK(cudaSetDevice(h->device));
    if (const int r = h->b_scratch.reserve(h, in.S); r != F1L_OK) return r;
    return launch_pipeline(h, stream, in, h->b_scratch, o, h->timing != 0);
}

int f1l_plan_batch_call_dev(f1l_handle h, const f1l_batch_call* b, void* stream) {
    PipeIn in;
    BatchOut o;
    const int r = batch_args(h, b, in, o);
    return r != F1L_OK ? r : plan_batch_dev_internal(h, in, o, (cudaStream_t)stream);
}

// the moving-opponent fields of a batch call's pipeline, checked
static int motion_args(const f1l_batch_call* b, const double* opp_vel, double v_min, PipeIn& in) {
    if (const int r = check_motion(b->max_opp, opp_vel, v_min); r != F1L_OK) return r;
    in.motion = true;
    in.opp_vel = b->max_opp > 0 ? opp_vel : nullptr;
    in.v_min = v_min;
    return F1L_OK;
}

int f1l_plan_batch_motion_dev(f1l_handle h, const f1l_batch_call* b, const double* opp_vel_dev, double v_min,
                              void* stream) {
    PipeIn in;
    BatchOut o;
    int r = batch_args(h, b, in, o);
    if (r == F1L_OK) r = motion_args(b, opp_vel_dev, v_min, in);
    return r != F1L_OK ? r : plan_batch_dev_internal(h, in, o, (cudaStream_t)stream);
}

int f1l_plan_batch_dev(f1l_handle h, const double* poses_dev, const double* opp_dev,
                       const int32_t* n_opp_dev, int S, int max_opp, int32_t* best_idx_dev,
                       float* best_cost_dev, float* best_traj_dev, float* costs_dev,
                       uint8_t* flags_dev, double* steer_speed_dev, void* stream) {
    return f1l_plan_batch_prev_dev(h, poses_dev, opp_dev, n_opp_dev, S, max_opp, nullptr, nullptr, 0,
                                   best_idx_dev, best_cost_dev, best_traj_dev, costs_dev, flags_dev,
                                   steer_speed_dev, stream);
}

int f1l_plan_batch_prev_dev(f1l_handle h, const double* poses_dev, const double* opp_dev,
                            const int32_t* n_opp_dev, int S, int max_opp, float* prev_theta_dev,
                            uint8_t* has_prev_dev, int update_prev, int32_t* best_idx_dev,
                            float* best_cost_dev, float* best_traj_dev, float* costs_dev,
                            uint8_t* flags_dev, double* steer_speed_dev, void* stream) {
    const f1l_batch_call b = {poses_dev, opp_dev, n_opp_dev, S, max_opp, prev_theta_dev, has_prev_dev,
                              update_prev, 0, nullptr, best_idx_dev, best_cost_dev, best_traj_dev,
                              costs_dev, flags_dev, steer_speed_dev, nullptr};
    return f1l_plan_batch_call_dev(h, &b, stream);
}

// `in` and `o` hold host pointers: each chunk is copied in, planned and copied back on a slot stream
static int plan_batch_internal(f1l_handle h, const PipeIn& in, const BatchOut& o) {
    CK(cudaSetDevice(h->device));
    const int S = in.S, C = in.span.C, M = h->cfg.n_samples;
    // chunked 3-stream pipeline: H2D(i+1) | kernels(i) | D2H(i-1)
    // 8192-scenario chunks (0.23 M candidates: 1 ms of kernels against ~30 us of launches) for
    // large batches; smaller batches are cut into about eight chunks, down to 1024 scenarios.  The
    // last chunks taper (half, quarter, ... of a chunk, down to 1024): the result copy of the final
    // chunk is the one transfer nothing overlaps, 14 MB at full size but under 2 MB tapered.
    int chunk = 8192;
    if (S < 8 * chunk) { chunk = (S + 7) / 8; if (chunk < 1024) chunk = 1024; }
    if (chunk > S) chunk = S;
    int slot = 0;
    for (int s0 = 0, n = 0; s0 < S; s0 += n, slot = (slot + 1) % N_PIPE) {
        n = (S - s0 < chunk) ? (S - s0) : chunk;
        // rest = what is left after this chunk: keep halving while the tail is short
        const int rest = S - s0;
        if (rest < 2 * chunk && rest > 1024) { n = rest / 2; if (n < 1024) n = 1024; if (n > rest) n = rest; }
        NvtxRange nvtx_chunk("f1l.plan_batch.chunk (H2D, kernels, D2H)");
        PipeSlot& p = h->pipe[slot];
        cudaStream_t st = p.stream;
        CK(cudaStreamSynchronize(st));  // slot buffers free again (grow-only ensure below)
        if (const int r = p.scratch.reserve(h, n); r != F1L_OK) return r;
        // the chunk's arrays: the previous paths travel in and, with update_prev, back out
        const Stage t[B_ARRAYS] = {
            {&p.buf[B_POSES], in.poses, nullptr, 32},
            {&p.buf[B_OPP], in.opp, nullptr, (size_t)in.max_opp * 24},
            {&p.buf[B_NOPP], in.n_opp, nullptr, 4},
            {&p.buf[B_IDX], nullptr, o.best_idx, 4},
            {&p.buf[B_COST], nullptr, o.best_cost, 4},
            {&p.buf[B_TRAJ], nullptr, o.best_traj, (size_t)M * 16},
            {&p.buf[B_COSTS], nullptr, o.costs, (size_t)C * 4},
            {&p.buf[B_FLAGS], nullptr, o.flags, (size_t)C},
            {&p.buf[B_SS], nullptr, o.steer_speed, 16},
            {&p.buf[B_PREV], in.prev_theta, o.prev_out, (size_t)M * 4},
            {&p.buf[B_PVALID], in.prev_valid, o.prev_valid_out, 1},
            {&p.buf[B_W], in.weights, nullptr, F1L_N_TERMS * 4},
            {&p.buf[B_TERMS], nullptr, o.terms, (size_t)C * F1L_N_TERMS * 4},
            {&p.buf[B_VEL], in.opp_vel, nullptr, (size_t)in.max_opp * 16},
        };
        if (const int r = stage_in(h, st, t, s0, n); r != F1L_OK) return r;
        // the chunk is a batch call of n scenarios on the slot's copies (updated in place)
        f1l_batch_call d{};
        d.poses = (const double*)t[B_POSES].dev();
        d.opp = (const double*)t[B_OPP].dev();
        d.n_opp = (const int32_t*)t[B_NOPP].dev();
        d.n_scenarios = n;
        d.max_opp = in.max_opp;
        d.prev_theta = (float*)t[B_PREV].dev();
        d.has_prev = (uint8_t*)t[B_PVALID].dev();
        d.update_prev = o.prev_out != nullptr;
        d.weights = (const float*)t[B_W].dev();
        d.best_idx = (int32_t*)t[B_IDX].dev();
        d.best_cost = (float*)t[B_COST].dev();
        d.best_traj = (float*)t[B_TRAJ].dev();
        d.costs = (float*)t[B_COSTS].dev();
        d.flags = (uint8_t*)t[B_FLAGS].dev();
        d.steer_speed = (double*)t[B_SS].dev();
        d.terms = (float*)t[B_TERMS].dev();
        PipeIn din;
        BatchOut dout;
        int r = batch_args(h, &d, din, dout);
        if (r == F1L_OK && in.motion) r = motion_args(&d, (const double*)t[B_VEL].dev(), in.v_min, din);
        if (r == F1L_OK) r = launch_pipeline(h, st, din, p.scratch, dout, false);
        if (r == F1L_OK) r = stage_out(h, st, t, s0, n);
        if (r != F1L_OK) return r;
    }
    for (int i = 0; i < N_PIPE; ++i) CK(cudaStreamSynchronize(h->pipe[i].stream));
    return F1L_OK;
}

int f1l_plan_batch_call(f1l_handle h, const f1l_batch_call* b) {
    PipeIn in;
    BatchOut o;
    const int r = batch_args(h, b, in, o);
    return r != F1L_OK ? r : plan_batch_internal(h, in, o);
}

int f1l_plan_batch_motion(f1l_handle h, const f1l_batch_call* b, const double* opp_vel, double v_min) {
    PipeIn in;
    BatchOut o;
    int r = batch_args(h, b, in, o);
    if (r == F1L_OK) r = motion_args(b, opp_vel, v_min, in);
    if (r != F1L_OK) return r;
    // a NaN velocity would silently clear a collision: every velocity in use must be finite
    for (int s = 0; s < b->n_scenarios; ++s) {
        int k_n = b->n_opp ? b->n_opp[s] : b->max_opp;
        k_n = k_n < 0 ? 0 : (k_n > b->max_opp ? b->max_opp : k_n);
        for (int k = 0; k < 2 * k_n; ++k)
            if (!std::isfinite(opp_vel[2 * (size_t)s * b->max_opp + k])) return F1L_ERR_INVALID_ARG;
    }
    return plan_batch_internal(h, in, o);
}

int f1l_plan_batch(f1l_handle h, const double* poses, const double* opp, const int32_t* n_opp,
                   int S, int max_opp, int32_t* best_idx, float* best_cost, float* best_traj,
                   float* costs, uint8_t* flags, double* steer_speed) {
    return f1l_plan_batch_prev(h, poses, opp, n_opp, S, max_opp, nullptr, nullptr, 0, best_idx, best_cost,
                               best_traj, costs, flags, steer_speed);
}

int f1l_plan_batch_prev(f1l_handle h, const double* poses, const double* opp, const int32_t* n_opp,
                        int S, int max_opp, float* prev_theta, uint8_t* has_prev, int update_prev,
                        int32_t* best_idx, float* best_cost, float* best_traj, float* costs,
                        uint8_t* flags, double* steer_speed) {
    const f1l_batch_call b = {poses, opp, n_opp, S, max_opp, prev_theta, has_prev, update_prev, 0, nullptr,
                              best_idx, best_cost, best_traj, costs, flags, steer_speed, nullptr};
    return f1l_plan_batch_call(h, &b);
}

// ---- closed-loop rollouts -----------------------------------------------------------------
int f1l_default_rollout_config(f1l_rollout_config* rc) {
    if (!rc) return F1L_ERR_INVALID_ARG;
    rc->dt = 0.01;
    rc->substeps = 1;
    rc->group = 1;
    rc->max_steer = 0.4189;
    rc->max_accel = 9.51;
    rc->v_max = INFINITY;
    return F1L_OK;
}

int f1l_default_vehicle(f1l_vehicle* veh) {
    if (!veh) return F1L_ERR_INVALID_ARG;
    *veh = f1l_vehicle{1.0489, 4.718, 5.4562, 0.15875, 0.17145, 0.074, 3.74, 0.04712, 3.2, 7.319, 0.5};
    return F1L_OK;
}

// every rollout entry point: veh == nullptr runs the kinematic bicycle, else the single-track model
// on dyn (checked by the caller)
// predict: every step plans against the opponents' constant-velocity prediction (v_min checked)
static int rollout_internal(f1l_handle h, const f1l_rollout_config* rc, const f1l_vehicle* veh,
                            const f1l_fleet* fl, double* dyn, const float* weights_dev, int S, int n_steps,
                            const f1l_rollout_trace* trace, double* trace_dyn, void* stream,
                            bool predict = false, double v_min = 1.0) {
    if (!h || !rc || !fl) return F1L_ERR_INVALID_ARG;
    if (predict && (!std::isfinite(v_min) || !(v_min > 0.0))) return F1L_ERR_INVALID_ARG;
    if (!fl->state || !fl->prev_theta || !fl->has_prev || !fl->status || !fl->progress ||
        !fl->track_i || !fl->track_s)
        return F1L_ERR_INVALID_ARG;
    if (rc->group < 1 || rc->group > F1L_MAX_GROUP || S <= 0 || S % rc->group != 0) return F1L_ERR_INVALID_ARG;
    if (rc->substeps < 1 || n_steps < 0) return F1L_ERR_INVALID_ARG;
    if (!(rc->dt > 0) || !(rc->max_steer > 0) || !(rc->max_accel > 0) || !(rc->v_max > 0))
        return F1L_ERR_INVALID_ARG;
    if (n_steps == 0) return F1L_OK;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    PipeIn in;
    if (const int r = make_span(h, 0, Shard{}, false, in.span); r != F1L_OK) return r;
    CK(cudaSetDevice(h->device));
    ENS(h->r_ss, (size_t)S * 16);
    ENS(h->r_cost, (size_t)S * 4);
    ENS(h->r_opp, (size_t)S * F1L_MAX_OPP * 24);
    ENS(h->r_nopp, (size_t)S * 4);
    if (predict) ENS(h->r_vel, (size_t)S * F1L_MAX_OPP * 16);
    PipeScratch& sc = h->b_scratch;   // every step's pipeline reserves it for the same S: no realloc
    if (const int r = sc.reserve(h, S); r != F1L_OK) return r;
    cudaStream_t st = (cudaStream_t)stream;
    NvtxRange nvtx_rollout("f1l.rollout");

    RolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.tr = track_view(h);
    a.grid = grid_view(h);
    a.seg_s = (const double2*)h->seg_s.p;
    a.lap = h->lap;
    a.res = h->gres;
    a.has_grid = h->grid.p != nullptr;
    a.collision_mode = h->cfg.collision_mode;
    a.hl = 0.5 * h->cfg.car_length;
    a.hw = 0.5 * h->cfg.car_width;
    a.disc_off = h->cfg.car_length / 3.0;
    a.wheelbase = h->cfg.wheelbase;
    a.dt = rc->dt;
    a.max_steer = rc->max_steer;
    a.max_accel = rc->max_accel;
    a.v_max = rc->v_max;
    a.substeps = rc->substeps;
    a.group = rc->group;
    a.n_races = S / rc->group;
    a.state = fl->state;
    a.status = fl->status;
    a.progress = fl->progress;
    a.track_i = fl->track_i;
    a.track_s = fl->track_s;
    a.opp = (double*)h->r_opp.p;
    a.n_opp = (int32_t*)h->r_nopp.p;
    if (veh) {
        a.dyn = dyn;
        a.veh = *veh;
    }
    a.opp_vel = predict ? (double*)h->r_vel.p : nullptr;
    void (*const step)(RolloutArgs) = veh ? rollout_step_kernel<SingleTrack> : rollout_step_kernel<Kinematic>;
    const unsigned blocks = (unsigned)((a.n_races + ROLLOUT_WARPS - 1) / ROLLOUT_WARPS);

    // once per call: global nearest_point of every car (K1) for the cars to re-acquire, then the
    // initial pass of the step kernel (no integration) builds step 0's opponent table.  Both run
    // in the batch scratch: they are enqueued before the first step's pipeline overwrites it.
    PPOut po{};
    po.nearest = (double*)sc.near4.p;
    po.nearest_i = (int32_t*)sc.near_i.p;
    launch_pp(h, st, fl->state, 4, S, -1.0, h->cfg.wheelbase, 0.0, 0, 0.0, (unsigned long long*)sc.best.p, po);
    a.near_i = po.nearest_i;
    a.near4 = po.nearest;
    step<<<blocks, ROLLOUT_WARPS * 32, 0, st>>>(a);
    h->launches += 3;
    CK(cudaGetLastError());
    a.near_i = nullptr;
    a.near4 = nullptr;
    a.steer_speed = (const double*)h->r_ss.p;
    a.best_cost = (const float*)h->r_cost.p;
    // every step plans the fleet as f1l_plan_batch_call_dev does with update_prev and these weights
    in.poses = fl->state;
    in.opp = a.opp;
    in.n_opp = a.n_opp;
    in.S = S;
    in.max_opp = F1L_MAX_OPP;
    in.prev_theta = fl->prev_theta;
    in.prev_stride = h->cfg.n_samples;
    in.prev_valid = fl->has_prev;
    in.weights = weights_dev;
    if (predict) {
        in.motion = true;
        in.opp_vel = a.opp_vel;
        in.v_min = v_min;
    }
    BatchOut o;
    o.best_cost = (float*)h->r_cost.p;
    o.steer_speed = (double*)h->r_ss.p;
    o.prev_out = fl->prev_theta;
    o.prev_valid_out = fl->has_prev;
    for (int k = 0; k < n_steps; ++k) {
        const size_t row = (size_t)k * S;
        o.best_idx = trace && trace->best_idx ? trace->best_idx + row : nullptr;
        if (const int r = plan_batch_dev_internal(h, in, o, st); r != F1L_OK) return r;
        a.tr_state = trace && trace->state ? trace->state + 4 * row : nullptr;
        a.tr_ss = trace && trace->steer_speed ? trace->steer_speed + 2 * row : nullptr;
        a.tr_status = trace && trace->status ? trace->status + row : nullptr;
        a.tr_progress = trace && trace->progress ? trace->progress + row : nullptr;
        a.tr_dyn = trace_dyn ? trace_dyn + 3 * row : nullptr;
        step<<<blocks, ROLLOUT_WARPS * 32, 0, st>>>(a);
        h->launches += 1;
        CK(cudaGetLastError());
    }
    return F1L_OK;
}

int f1l_rollout_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_fleet* fl, int S,
                    int n_steps, const f1l_rollout_trace* trace, void* stream) {
    return rollout_internal(h, rc, nullptr, fl, nullptr, nullptr, S, n_steps, trace, nullptr, stream);
}

int f1l_rollout_weights_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_fleet* fl,
                            const float* weights_dev, int S, int n_steps, const f1l_rollout_trace* trace,
                            void* stream) {
    return rollout_internal(h, rc, nullptr, fl, nullptr, weights_dev, S, n_steps, trace, nullptr, stream);
}

static int check_vehicle(const f1l_vehicle* veh, const double* dyn_dev) {
    if (!veh || !dyn_dev) return F1L_ERR_INVALID_ARG;
    for (const double p : {veh->mu, veh->C_Sf, veh->C_Sr, veh->lf, veh->lr, veh->m, veh->I, veh->max_steer_vel,
                           veh->v_switch, veh->v_kin})
        if (!(p > 0)) return F1L_ERR_INVALID_ARG;
    if (!(veh->h >= 0)) return F1L_ERR_INVALID_ARG;
    return F1L_OK;
}

int f1l_rollout_st_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_vehicle* veh,
                       const f1l_fleet* fl, double* dyn_dev, const float* weights_dev, int S, int n_steps,
                       const f1l_rollout_trace* trace, double* trace_dyn_dev, void* stream) {
    if (const int r = check_vehicle(veh, dyn_dev); r != F1L_OK) return r;
    return rollout_internal(h, rc, veh, fl, dyn_dev, weights_dev, S, n_steps, trace, trace_dyn_dev, stream);
}

int f1l_rollout_predict_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_vehicle* veh,
                            const f1l_fleet* fl, double* dyn_dev, const float* weights_dev, double v_min,
                            int S, int n_steps, const f1l_rollout_trace* trace, double* trace_dyn_dev,
                            void* stream) {
    if (veh)
        if (const int r = check_vehicle(veh, dyn_dev); r != F1L_OK) return r;
    return rollout_internal(h, rc, veh, fl, veh ? dyn_dev : nullptr, weights_dev, S, n_steps, trace,
                            veh ? trace_dyn_dev : nullptr, stream, true, v_min);
}

// ---- pure pursuit -------------------------------------------------------------------------
int f1l_pure_pursuit_batch_dev(f1l_handle h, const double* poses_dev, int n_poses, double L,
                               double* nearest_dev, int32_t* nearest_i_dev, double* lookahead_dev,
                               int32_t* lookahead_i_dev, double* actuation_dev,
                               int32_t* status_dev, void* stream) {
    if (!h || !poses_dev || n_poses <= 0) return F1L_ERR_INVALID_ARG;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    CK(cudaSetDevice(h->device));
    NvtxRange nvtx_pp("f1l.pure_pursuit_batch (K1 scan + finish)");
    PPOut o{};
    o.nearest = nearest_dev;
    o.nearest_i = nearest_i_dev;
    o.lookahead = lookahead_dev;
    o.lookahead_i = lookahead_i_dev;
    o.actuation = actuation_dev;
    o.status = status_dev;
    ENS(h->pp_key, (size_t)n_poses * 8);   // scan scratch (one call in flight per handle)
    launch_pp(h, (cudaStream_t)stream, poses_dev, 3, n_poses, L, h->cfg.wheelbase, h->cfg.max_reacquire, 0,
              0.0, (unsigned long long*)h->pp_key.p, o);
    h->launches += 2;
    CK(cudaGetLastError());
    return F1L_OK;
}

int f1l_pure_pursuit_batch(f1l_handle h, const double* poses, int n, double L, double* nearest,
                           int32_t* nearest_i, double* lookahead, int32_t* lookahead_i,
                           double* actuation, int32_t* status) {
    if (!h || !poses || n <= 0) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const Stage t[] = {{&h->m[0], poses, nullptr, 24},       {&h->m[1], nullptr, nearest, 32},
                       {&h->m[2], nullptr, nearest_i, 4},    {&h->m[3], nullptr, lookahead, 32},
                       {&h->m[4], nullptr, lookahead_i, 4},  {&h->m[5], nullptr, actuation, 16},
                       {&h->m[6], nullptr, status, 4}};
    int r = stage_in(h, st, t, 0, n);
    if (r == F1L_OK)
        r = f1l_pure_pursuit_batch_dev(h, (const double*)t[0].dev(), n, L, (double*)t[1].dev(),
                                       (int32_t*)t[2].dev(), (double*)t[3].dev(), (int32_t*)t[4].dev(),
                                       (double*)t[5].dev(), (int32_t*)t[6].dev(), st);
    if (r == F1L_OK) r = stage_out(h, st, t, 0, n);
    if (r != F1L_OK) return r;
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

int f1l_front_axle_batch_dev(f1l_handle h, const double* poses_dev, int n_poses, double wheelbase,
                             double k_path, double* front_dev, int32_t* nearest_i_dev,
                             void* stream) {
    if (!h || !poses_dev || n_poses <= 0 || !front_dev) return F1L_ERR_INVALID_ARG;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    CK(cudaSetDevice(h->device));
    PPOut o{};
    o.nearest_i = nearest_i_dev;
    o.front = front_dev;
    ENS(h->pp_key, (size_t)n_poses * 8);
    launch_pp(h, (cudaStream_t)stream, poses_dev, 4, n_poses, 0.0, wheelbase, 0.0, 1, k_path,
              (unsigned long long*)h->pp_key.p, o);
    h->launches += 2;
    CK(cudaGetLastError());
    return F1L_OK;
}

int f1l_front_axle_batch(f1l_handle h, const double* poses, int n, double wheelbase, double k_path,
                         double* front, int32_t* nearest_i) {
    if (!h || !poses || n <= 0 || !front) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const Stage t[] = {{&h->m[0], poses, nullptr, 32}, {&h->m[1], nullptr, front, 48},
                       {&h->m[2], nullptr, nearest_i, 4}};
    int r = stage_in(h, st, t, 0, n);
    if (r == F1L_OK)
        r = f1l_front_axle_batch_dev(h, (const double*)t[0].dev(), n, wheelbase, k_path, (double*)t[1].dev(),
                                     (int32_t*)t[2].dev(), st);
    if (r == F1L_OK) r = stage_out(h, st, t, 0, n);
    if (r != F1L_OK) return r;
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

int f1l_intersect_point_batch(f1l_handle h, const double* points, const double* t_start, int n,
                              double radius, int wrap, double* out, int32_t* out_i) {
    if (!h || !points || !t_start || n <= 0 || !out || !out_i) return F1L_ERR_INVALID_ARG;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    // the scan indexes waypoint int(t) and its wrap loop reduces indices in [-1, int(t)] with one
    // conditional add: start parameters outside [0, N) (or NaN) would read out of bounds
    for (int i = 0; i < n; ++i)
        if (!(t_start[i] >= 0.0 && t_start[i] < (double)h->n)) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const Stage t[] = {{&h->m[0], points, nullptr, 16}, {&h->m[1], t_start, nullptr, 8},
                       {&h->m[2], nullptr, out, 32}, {&h->m[3], nullptr, out_i, 4}};
    if (const int r = stage_in(h, st, t, 0, n); r != F1L_OK) return r;
    intersect_batch_kernel<<<(n + 63) / 64, 64, 0, st>>>(
        track_view(h), (const double*)t[0].dev(), (const double*)t[1].dev(), n, radius, wrap,
        (double*)t[2].dev(), (int32_t*)t[3].dev());
    h->launches += 1;
    CK(cudaGetLastError());
    if (const int r = stage_out(h, st, t, 0, n); r != F1L_OK) return r;
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

int f1l_get_actuation_batch(f1l_handle h, const double* in, int n, double wheelbase, double* out) {
    if (!h || !in || n <= 0 || !out) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const Stage t[] = {{&h->m[0], in, nullptr, 56}, {&h->m[1], nullptr, out, 16}};
    if (const int r = stage_in(h, st, t, 0, n); r != F1L_OK) return r;
    actuation_batch_kernel<<<(n + 63) / 64, 64, 0, st>>>((const double*)t[0].dev(), n, wheelbase,
                                                         (double*)t[1].dev());
    h->launches += 1;
    CK(cudaGetLastError());
    if (const int r = stage_out(h, st, t, 0, n); r != F1L_OK) return r;
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

// debug: the last single query's context (teacher-forced collision tests):
// out[0..1] cos/sin pose, [2..7] grid A00 A01 A10 A11 fx fy, [8..9] gix giy (as float bits via
// int copy), [10..] opponents 16 x (x, y, cos, sin)
int f1l_debug_query_ctx(f1l_handle h, float* out_f, int32_t* out_i) {
    if (!h || !out_f || !out_i || !h->q_scratch.ctx.p) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    QueryCtx q;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(&q, h->q_scratch.ctx.p, sizeof(q), cudaMemcpyDeviceToHost));
    out_f[0] = q.cth; out_f[1] = q.sth;
    out_f[2] = q.gA00; out_f[3] = q.gA01; out_f[4] = q.gA10; out_f[5] = q.gA11;
    out_f[6] = q.gfx; out_f[7] = q.gfy;
    for (int k = 0; k < F1L_MAX_OPP; ++k) {
        const float4 o = k < q.n_opp ? q.opp[k] : make_float4(1e9f, 1e9f, 1.0f, 0.0f);   // unused: far away
        out_f[8 + 4 * k] = o.x; out_f[9 + 4 * k] = o.y;
        out_f[10 + 4 * k] = o.z; out_f[11 + 4 * k] = o.w;
    }
    out_i[0] = q.gix; out_i[1] = q.giy; out_i[2] = q.i_ego; out_i[3] = q.seg0;
    out_i[4] = q.nseg; out_i[5] = q.n_opp;
    return F1L_OK;
}

// NUMA node of a CUDA device from sysfs (PCI bus id -> /sys/bus/pci/devices/<id>/numa_node), then
// the calling thread's CPU affinity := that node's CPUs (/sys/devices/system/node/nodeN/cpulist).
int f1l_bind_host_numa(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return F1L_ERR_NO_DEVICE;
    for (char* c = bus; *c; ++c) if (*c >= 'A' && *c <= 'Z') *c = (char)(*c - 'A' + 'a');
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -100;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return -100;   // the platform does not say (single node / VM): nothing to do
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return -100;
    cpu_set_t set;
    CPU_ZERO(&set);
    int lo = 0, hi = 0, n = 0;
    for (;;) {   // "0-15,64-79"
        if (fscanf(f, "%d", &lo) != 1) break;
        hi = lo;
        int c = fgetc(f);
        if (c == '-') { if (fscanf(f, "%d", &hi) != 1) break; c = fgetc(f); }
        for (int k = lo; k <= hi && k < CPU_SETSIZE; ++k) { CPU_SET(k, &set); ++n; }
        if (c != ',') break;
    }
    fclose(f);
    if (n == 0) return -100;
    // keep only CPUs this process may use at all (cgroup / taskset limits)
    cpu_set_t cur;
    if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {
        cpu_set_t both;
        CPU_AND(&both, &set, &cur);
        if (CPU_COUNT(&both) == 0) return -100;
        set = both;
    }
    if (sched_setaffinity(0, sizeof(set), &set) != 0) return -100;
    return node;
}

int f1l_measure_peaks(f1l_handle h, double* fp32_tflops, double* mufu_gops) {
    if (!h) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    ENS(h->m[0], (size_t)h->sm_count * 8 * 256 * 4);
    cudaStream_t st = h->stream;
    const int blocks = h->sm_count * 8, threads = 256, iters = 4096;
    float ms = 0.f;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        ffma_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m[0].p, iters, 1.0001f, 0.5f);
        CK(cudaEventRecord(h->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    }
    h->launches += 3;
    if (fp32_tflops)
        *fp32_tflops = 2.0 * PEAK_CHAINS * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        mufu_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m[0].p, iters);
        CK(cudaEventRecord(h->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    }
    h->launches += 3;
    if (mufu_gops)
        *mufu_gops = (double)PEAK_CHAINS * iters * blocks * threads / (ms * 1e-3) / 1e9;
    CK(cudaGetLastError());
    return F1L_OK;
}

// extended pipe probes: out[0] FFMA TFLOP/s, out[1] MUFU Gop/s, out[2] packed FFMA2 TFLOP/s,
// out[3] warp-instructions per clock per SM of an 8 FFMA + 8 FMNMX mix (shared issue slot probe)
int f1l_measure_peaks_ex(f1l_handle h, double* out, int n) {
    if (!h || !out || n < 4) return F1L_ERR_INVALID_ARG;
    int r = f1l_measure_peaks(h, &out[0], &out[1]);
    if (r != F1L_OK) return r;
    cudaStream_t st = h->stream;
    const int blocks = h->sm_count * 8, threads = 256, iters = 4096;
    float ms = 0.f;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        ffma2_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m[0].p, iters, 1.0001f, 0.5f);
        CK(cudaEventRecord(h->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    }
    out[2] = 4.0 * PEAK_CHAINS * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        mixed_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m[0].p, iters, 1.0001f, 0.5f);
        CK(cudaEventRecord(h->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    }
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device);
    const double warp_inst = 16.0 * iters * (double)blocks * threads / 32.0;
    out[3] = warp_inst / (ms * 1e-3) / ((double)khz * 1e3) / h->sm_count;
    h->launches += 6;
    return F1L_OK;
}

}  // extern "C"
