// f1l_api.cu -- C-ABI (include/f1l.h) over the sm_100a kernels.  No torch types, no exceptions
// across the boundary; every launch goes on the handle's (or the caller's) stream.
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
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

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct PipeSlot {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    DevBuf poses, opp, nopp, ctx, centres, best, idx, cost, traj, costs, flags, ss, near_i, near4;
    DevBuf prev, pvalid;   // the chunk's previous paths [n,M] f32 and their flags [n] u8
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
    unsigned long long gkey[4] = {~0ull, ~0ull, ~0ull, ~0ull};
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
    DevBuf q_res, q_in, q_goals, q_ctx, q_centres, q_best, q_states, q_headings, q_params, q_flags;
    // pinned staging for the single query
    void* h_in = nullptr;   // pose + opponents
    void* h_out = nullptr;  // header + best trajectory
    void* h_out_dev = nullptr;  // the same block as the device sees it (mapped pinned memory): the
                                // select kernel of a single query writes its results straight into it
    size_t h_out_cap = 0;
    // per-candidate detail block of a single query (costs | terms | goals | params | flags): one
    // device block, one D2H into pinned staging, then plain copies into the caller's arrays
    DevBuf q_detail;
    void* h_detail = nullptr;
    size_t h_detail_cap = 0;
    // deviation-pass work counters (f1l_set_stats / f1l_get_stats)
    DevBuf stats;
    int stats_on = 0;
    // batch (device-pointer API) scratch
    DevBuf b_ctx, b_centres, b_best, b_near_i, b_near4;
    // rollout (f1l_rollout_dev) scratch: command, cost, the races' opponent table, re-acquisition
    DevBuf r_ss, r_cost, r_opp, r_nopp, r_key, r_near_i, r_near4;
    // batch pipeline (host-pointer API)
    PipeSlot pipe[N_PIPE];
    // misc scratch for the pure-pursuit / intersect host APIs
    DevBuf m_in, m_in2, m_o0, m_o1, m_o2, m_o3, m_o4, m_o5, pp_key;
    // peer-memory exchange of candidate-sharded queries (f1l_xchg_*): the local block, the peers'
    // blocks as mapped by cudaIpcOpenMemHandle (own rank: the local pointer)
    int pp_per_sm = 0, pp_per_sm_ct = 0;   // resident pp_scan_kernel CTAs per SM (pp_slots): global / constant table
    unsigned long long ctab_key = 0;   // != 0: this handle's track sits in the constant-memory table
                                       // (as long as it is still the device's owner, ctab_owner)
    DevBuf xchg;
    XchgView xview = {0, 0, {nullptr}};
    // template instance / CTA plan of the last eval_kernel launch (f1l_last_eval_shape)
    int eval_info[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // the last single query, for f1l_select_candidate: candidate count, explicit goals?, epoch
    int lastq_C = 0, lastq_goals = 0;
    int lastq_rows[3] = {0, 1, -1};   // lookahead rows its sampler filled (row0, step, count; -1: all)
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

void release(DevBuf& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

#define ENS(buf, bytes)                          \
    do {                                         \
        int r__ = ensure(h, (buf), (bytes));     \
        if (r__ != F1L_OK) return r__;           \
    } while (0)

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

// One compiled eval_kernel: the resident CTAs per SM its register budget is built for (MINB), and
// its shared memory in front of the window table (EvalSmem::C_TAB).
struct EvalBuild {
    eval_fn fn;   // null: not built
    int minb;
    uint32_t smem_fixed;
    size_t smem_bytes(int nseg_pad) const {
        return smem_fixed + (size_t)(nseg_pad + EVAL_SEG_PAD) * (2 * sizeof(float4));
    }
};

// The kernels that serve sample counts M <= m_max: the deviation-pass shape (IPL samples per lane;
// S samples per lane x SG sample groups in the loop), one eval build per warp count, and the select
// and generate kernels of the same IPL.
struct EvalBucket {
    int m_max, ipl, s, sg;
    EvalBuild nw4, nw7, nw8;
    EvalBuild wide;   // 8 warps at two CTAs per SM (128 registers), large dense queries
    select_fn select;
    generate_fn generate;
    const EvalBuild& build(int nw) const { return nw == 4 ? nw4 : (nw == 7 ? nw7 : nw8); }
};

template <int IPL, int S, int SG, int NW, int MINB>
EvalBuild eval_build() {
    if constexpr (MINB == 0) return {nullptr, 0, 0};
    else return {eval_kernel<IPL, S, SG, NW, MINB>, MINB, EvalSmem<S, SG, NW>::C_TAB};
}
template <int M_MAX, int IPL, int S, int SG, int MINB4, int MINB7, int MINB8, int MINB_WIDE>
EvalBucket eval_bucket() {
    return {M_MAX, IPL, S, SG,
            eval_build<IPL, S, SG, 4, MINB4>(), eval_build<IPL, S, SG, 7, MINB7>(),
            eval_build<IPL, S, SG, 8, MINB8>(), eval_build<IPL, S, SG, 8, MINB_WIDE>(),
            select_kernel<IPL>, generate_kernel<IPL>};
}

// Every eval_kernel instance and its residency, one row per bucket (MINB 0: no such build).
// NW = 7 (four resident CTAs of 7 warps at <= 72 registers) serves candidate counts that are a
// small multiple of 7 -- the default 4x7 goal grid; everything else runs 8-warp CTAs (three at 80).
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
    eval_bucket<     208,   7, 13, 16,   7, 4, 3, 2>(),
    eval_bucket<F1L_MAX_M,  8, 16, 16,   7, 4, 3, 2>(),
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
    // tuning hook for experiments: F1L_EVAL_PLAN="<warps>,<candidates per CTA>"
    if (const char* e = getenv("F1L_EVAL_PLAN")) {
        int nw = 0, chunk = 0;
        if (sscanf(e, "%d,%d", &nw, &chunk) == 2 && (nw == 4 || nw == 7 || nw == 8) && chunk >= nw &&
            chunk % nw == 0 && !(nw != 8 && M > 128))
            return CtaPlan{nw, chunk, (n_cand + chunk - 1) / chunk};
    }
    // Throughput regime -- many waves of small scenarios (the 4x7 grid: 28 candidates) with shared
    // Newton solves: one 4-warp CTA per scenario whose warps pull the scenario's 4-candidate items.
    // Measured, not modelled (the wave model below counts CTAs and would always prefer the CTA with
    // more warps at equal residency): 10.84 ms on the bench workload against 11.19 for 7-warp CTAs.
    {
        const int full4 = ((n_cand + 3) / 4) * 4;
        if (cubic && M <= 128 && full4 >= 4 * EVAL_ITEM && n_cand <= 256 &&
            (long long)S >= 8LL * eval_bucket_of(M).nw4.minb * sm_count)
            return CtaPlan{4, full4, 1};
    }
    const int nws[3] = {4, 7, 8};
    for (int nw : nws) {
        if (nw != 8 && M > 128) continue;   // the 72-register builds of the M = 200 shapes spill
        const int resident = eval_bucket_of(M).build(nw).minb * sm_count;
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

// K1 = key preset + scan + finish on one stream.  key: 8 bytes of scratch per pose; slots: one-warp
// scan CTAs resident on the device (pp_slots)
void launch_pp(const TrackView& tv, cudaStream_t stream, const double* poses, int pose_stride,
               int n_poses, double L, double wb, double max_reacquire, int front_axle, double k_path,
               unsigned long long* key, int slots, const PPOut& o, bool ctab, f1l_handle owner = nullptr) {
    const int n_groups = (n_poses + PP_CTA_POSES - 1) / PP_CTA_POSES;
    const int nblk = (tv.n - 1 + 31) >> 5;
    int n_parts = pp_task_parts(n_groups, nblk, slots, ctab ? 16 : 6);
    if (const char* e = getenv("F1L_PP_PARTS")) {   // tuning hook
        const int v = atoi(e);
        if (v >= 1 && v <= PP_MAX_PARTS && v <= nblk) n_parts = v;
    }
    cudaMemsetAsync(key, 0xff, (size_t)n_poses * 8, stream);
    PPParts parts;
    parts.n = n_parts;
    parts.per = nblk / n_parts;
    parts.rem = nblk - parts.per * n_parts;
    const dim3 grid((unsigned)n_groups, (unsigned)n_parts);
    if (ctab) {
        std::lock_guard<std::mutex> lk(g_ctab_mu);
        ctab = owner && ctab_valid(owner);   // still ours?  (checked and enqueued under the mutex)
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
    int row0 = 0, row_step = 1;        // row-interleaved shard (c_begin / c_end are shard-local)
    const XchgView* xc = nullptr;      // sharded single query: exchange the argmin with the peers
    int32_t* xchg_status = nullptr;
    int s_row0 = 0, s_step = 1, s_rows = -1;   // lookahead rows the sampler must fill (-1: all)
    bool empty_shard = false;          // this rank owns no candidate of the query: it evaluates nothing
                                       // but still takes part in the exchange (key = ~0)
    int* work_next = nullptr;          // single query: device counter for the persistent-grid schedule
};

// select_kernel arguments of a pipeline over S scenarios (first_cand: the first evaluated candidate,
// returned when nothing at all was evaluated)
SelectArgs select_args(f1l_handle h, const TrackView& tv, const LutView& lut, const EvalParams& ep,
                       const QueryCtx* ctx, const Centre* centres, const float4* goals, int C,
                       int first_cand, const unsigned long long* best, int S, const BatchOut& o) {
    SelectArgs se;
    if (o.xc && S == 1) se.xc = *o.xc;
    else { se.xc.world = 0; se.xc.rank = 0; }
    se.xchg_status = o.xchg_status;
    se.tr = tv;
    se.lut = lut;
    se.ep = ep;
    se.ctx = ctx;
    se.centres = centres;
    se.widths = (const float*)h->widths.p;
    se.nL = h->nL;
    se.nW = h->nW;
    se.inv_nW = 1.0f / (float)(h->nW > 0 ? h->nW : 1);
    se.row0 = o.s_rows >= 0 ? o.s_row0 : 0;
    se.row_step = o.s_rows >= 0 ? o.s_step : 1;
    se.n_rows = o.s_rows >= 0 ? o.s_rows : h->nL;
    se.goals = goals;
    se.C = C;
    se.c_begin = first_cand < C ? first_cand : 0;   // (a rank without rows)
    se.best = best;
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

// sampler -> eval -> select for S scenarios on `stream`; all pointers are device pointers.
// Previous paths: scenario s reads prev_theta + s * prev_stride (stride 0: one path for all) when
// prev_valid is null or prev_valid[s] != 0; prev_theta null: no similarity term.
int launch_pipeline(f1l_handle h, cudaStream_t stream, const double* poses, const double* opp,
                    const int32_t* n_opp, int S, int max_opp, const float4* goals, int n_goals,
                    int c_begin, int c_end, QueryCtx* ctx, Centre* centres,
                    unsigned long long* best, int32_t* near_i, double* near4,
                    const float* prev_theta, int prev_stride, const uint8_t* prev_valid,
                    const BatchOut& o, bool time_it) {
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    const int C = goals ? n_goals : h->nL * h->nW;
    if (C <= 0) return F1L_ERR_NO_GOALS;
    if (c_begin < 0) c_begin = 0;
    if (o.empty_shard) { c_begin = 0; c_end = 0; }
    else {
        if (c_end <= 0 || c_end > C) c_end = C;
        if (c_begin >= c_end) return F1L_ERR_INVALID_ARG;
    }
    if (max_opp > F1L_MAX_OPP || max_opp < 0) return F1L_ERR_INVALID_ARG;
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
    const int n_cand = o.empty_shard ? 1 : c_end - c_begin;
    const CtaPlan cp = plan_ctas(n_cand, S, M, h->sm_count, ep.generator == 0);
    const int wpc = cp.nw;
    const EvalBucket& bucket = eval_bucket_of(M);
    const EvalBuild* build = &bucket.build(wpc);
    // A lone dense query that needs more than one wave of CTAs runs on a PERSISTENT grid instead: one
    // wave of CTAs whose warps pull single candidates from a device-wide counter, far lookahead rows
    // (the expensive candidates) first.  No wave quantisation, one window-table prologue per
    // resident CTA, and the cheap early-exit candidates fill the tail.
    int resident_ctas = build->minb * h->sm_count;
    // F1L_EVAL_DYNAMIC: 0 = never, 2 = whenever the query has more than one CTA (sanitizer runs at
    // small sizes), default = when it needs more than one wave
    static const int dyn_mode = getenv("F1L_EVAL_DYNAMIC") ? atoi(getenv("F1L_EVAL_DYNAMIC")) : 1;
    const bool dyn = S == 1 && wpc != 4 && o.work_next && !o.empty_shard && dyn_mode != 0 &&
                     ((long long)cp.ctas_per_scn > resident_ctas || (dyn_mode == 2 && cp.ctas_per_scn > 1));
    // ... and with at least F1L_EVAL_WIDE_MIN (default 4) candidates per resident warp it runs the
    // 128-register build of the M > 128 shapes on two CTAs per SM (measured on config 5: 65 536
    // candidates 471 -> 431 us, 32 768: 247 -> 234, 16 384: 134 -> 128, 8 192: 76 -> 100)
    static const int wide_min = getenv("F1L_EVAL_WIDE_MIN") ? atoi(getenv("F1L_EVAL_WIDE_MIN")) : 4;
    const bool wide = dyn && wpc == 8 && bucket.wide.fn && wide_min > 0 &&
                      (long long)n_cand >= (long long)wide_min * resident_ctas * wpc;
    if (wide) {
        build = &bucket.wide;
        resident_ctas = build->minb * h->sm_count;
    }
    const size_t smem = build->smem_bytes(nseg_pad);
    if (smem > 226 * 1024) return F1L_ERR_TOO_LARGE;

    SampleArgs sa;
    sa.tr = track_view(h);
    sa.grid = grid_view(h);
    sa.ep = ep;
    sa.poses = poses;
    sa.opp = opp;
    sa.n_opp = n_opp;
    sa.max_opp = max_opp;
    sa.lookaheads = (const double*)h->lookaheads.p;
    sa.nL = goals ? 0 : h->nL;
    sa.row0 = o.s_rows >= 0 ? o.s_row0 : 0;
    sa.row_step = o.s_rows >= 0 ? o.s_step : 1;
    sa.n_rows = o.s_rows >= 0 ? o.s_rows : h->nL;
    sa.ctx = ctx;
    sa.centres = centres;
    sa.best = best;
    sa.work_next = dyn ? o.work_next : nullptr;
    cudaEvent_t* ev = h->ev + 4 * h->ev_next;
    if (time_it) cudaEventRecord(ev[0], stream);
    nvtxRangePushA("f1l.sample");
    if (near_i && near4 && S >= 32) {
        // batch: nearest_point of all scenarios by the thread-per-pose scan kernel (K1), then one
        // warp per scenario for the lookahead intersections / context
        PPOut po;
        po.nearest = near4;
        po.nearest_i = near_i;
        po.lookahead = nullptr;
        po.lookahead_i = nullptr;
        po.actuation = nullptr;
        po.status = nullptr;
        po.front = nullptr;
        launch_pp(sa.tr, stream, poses, 4, S, -1.0, 0.33, 0.0, 0, 0.0, best, pp_slots(h), po, ctab_valid(h), h);   // `best` doubles as K1's key scratch: the sampler resets it
        sample_warp_kernel<<<(S + SAMPLE_WARPS - 1) / SAMPLE_WARPS, SAMPLE_WARPS * 32, 0, stream>>>(
            sa, near_i, near4, S);
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
    ea.goals = goals;
    ea.prev_theta = prev_theta;
    ea.prev_stride = prev_stride;
    ea.prev_valid = prev_valid;
    ea.C = C;
    ea.c_begin = c_begin;
    ea.c_end = c_end;
    ea.row0 = o.row0;
    ea.row_step = o.row_step > 1 ? o.row_step : 1;
    ea.chunk = cp.chunk;
    ea.ctas_per_scn = cp.ctas_per_scn;
    // four candidates per warp at a time (shared Newton) when every warp has at least four
    ea.item = (ep.generator == 0 && cp.chunk >= 4 * cp.nw) ? EVAL_ITEM : 1;
    ea.work_next = nullptr;
    ea.v_last = 0;
    if (dyn) {
        ea.work_next = o.work_next;
        ea.v_last = c_begin + c_end - 1;
        // single candidates per pull, unless every warp has at least four 4-candidate items to go
        // through: then the shared Newton solve pays more than the coarser tail costs
        ea.item = (ep.generator == 0 && (long long)n_cand >= 16LL * resident_ctas * wpc) ? EVAL_ITEM : 1;
        ea.ctas_per_scn = cp.ctas_per_scn < resident_ctas ? cp.ctas_per_scn : resident_ctas;
    }
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
    const long long n_ctas = (long long)S * ea.ctas_per_scn;
    if (n_ctas > 0x7fffffffLL) return F1L_ERR_TOO_LARGE;
    if (!o.empty_shard) build->fn<<<(unsigned)n_ctas, wpc * 32, smem, stream>>>(ea);
    {
        const int info[8] = {bucket.ipl, bucket.s, bucket.sg, wpc, build->minb, ea.chunk, ea.ctas_per_scn, ea.item};
        for (int i = 0; i < 8; ++i) h->eval_info[i] = info[i];
    }
    if (time_it) cudaEventRecord(ev[2], stream);

    const SelectArgs se = select_args(h, sa.tr, ea.lut, ep, ctx, centres, goals, C,
                                      o.row_step > 1 ? c_begin + o.row0 * h->nW : c_begin, best, S, o);
    bucket.select<<<S, SELECT_THREADS, 0, stream>>>(se);
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

// device / pinned-host result block of a single query: header then the best trajectory, so
// that one D2H copy brings everything a plain plan() call returns
struct QHeader {
    double steer, speed;                 // +0
    int32_t best_idx;                    // +16
    int32_t no_feasible, tracker_found;  // +20
    int32_t pad;                         // +28
    float best_cost;                     // +32
    float pad2[3];                       // -> 48 bytes, keeps the float4 trajectory 16-aligned
};
static_assert(sizeof(QHeader) == 48, "QHeader layout");
// result block: header | best trajectory float4[F1L_MAX_M] | map-frame trajectory double[F1L_MAX_M][4]
#define Q_OFF_TRAJ (sizeof(QHeader))
#define Q_OFF_MAP (Q_OFF_TRAJ + F1L_MAX_M * sizeof(float4))
#define Q_RES_BYTES (Q_OFF_MAP + F1L_MAX_M * 4 * sizeof(double))

// pinned-host / device input block of a single query (fixed size, so that the copy is a constant
// node of the CUDA graph): the opponent count travels in the block, not as a kernel argument
struct QInput {
    double pose[4];
    int32_t n_opp, pad;
    double opp[3 * F1L_MAX_OPP];
};

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
    if (!out || n < 4 || n_cand <= 0 || n_scenarios <= 0 || M < 2 || M > F1L_MAX_M || sm_count <= 0)
        return F1L_ERR_INVALID_ARG;
    const CtaPlan cp = plan_ctas(n_cand, n_scenarios, M, sm_count, generator == 0);
    out[0] = cp.nw;
    out[1] = cp.chunk;
    out[2] = cp.ctas_per_scn;
    out[3] = (generator == 0 && cp.chunk >= 4 * cp.nw) ? EVAL_ITEM : 1;
    return F1L_OK;
}

int f1l_debug_pp_parts(int n_poses, int n_waypoints, int slots) {
    if (n_poses <= 0 || n_waypoints < 2 || slots <= 0) return F1L_ERR_INVALID_ARG;
    return pp_task_parts((n_poses + PP_CTA_POSES - 1) / PP_CTA_POSES, (n_waypoints - 1 + 31) >> 5, slots);
}

int f1l_last_eval_shape(f1l_handle h, int32_t* out, int n) {
    if (!h || !out || n < 8) return F1L_ERR_INVALID_ARG;
    for (int i = 0; i < 8; ++i) out[i] = h->eval_info[i];
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
    for (int i = 0; i < N_PIPE && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&h->pipe[i].stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->pipe[i].done, cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaHostAlloc(&h->h_in, 1024, cudaHostAllocDefault);
    if (e == cudaSuccess) memset(h->h_in, 0, 1024);
    if (e == cudaSuccess) {
        h->h_out_cap = Q_RES_BYTES;
        e = cudaHostAlloc(&h->h_out, h->h_out_cap, cudaHostAllocMapped);
        if (e == cudaSuccess) {
            memset(h->h_out, 0, h->h_out_cap);
            static const bool direct_off = getenv("F1L_DIRECT_OUT") && atoi(getenv("F1L_DIRECT_OUT")) == 0;
            if (direct_off || cudaHostGetDevicePointer(&h->h_out_dev, h->h_out, 0) != cudaSuccess) {
                h->h_out_dev = nullptr;   // fall back to the device block + D2H copy
                cudaGetLastError();
            }
        }
    }
    if (e == cudaSuccess) {
        int sm = 0;
        cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
        if (sm > 0) h->sm_count = sm;
        // opt in to large dynamic shared memory for every eval instantiation
        const int big = 226 * 1024;  // opt-in maximum is 227 KB per block INCLUDING static shared memory
        for (const EvalBucket& b : kEvalBuckets) {
            for (const EvalBuild* eb : {&b.nw4, &b.nw7, &b.nw8, &b.wide}) {
                if (!eb->fn) continue;
                cudaError_t e2 = cudaFuncSetAttribute(eb->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, big);
                if (e2 != cudaSuccess && e == cudaSuccess) e = e2;
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
    release(h->xchg);
    DevBuf* bufs[] = {&h->xy, &h->v, &h->psi, &h->kappa, &h->segA, &h->segB, &h->blk, &h->grid, &h->clear, &h->clear_tmp, &h->edt,
                      &h->lut, &h->lookaheads, &h->widths, &h->prev, &h->q_res, &h->q_in, &h->q_goals,
                      &h->q_ctx, &h->q_centres, &h->q_best, &h->q_detail, &h->q_params, &h->q_flags, &h->q_states, &h->q_headings, &h->b_ctx, &h->b_centres,
                      &h->b_best, &h->b_near_i, &h->b_near4, &h->stats, &h->m_in, &h->m_in2, &h->m_o0, &h->m_o1, &h->m_o2, &h->m_o3,
                      &h->m_o4, &h->m_o5, &h->pp_key, &h->seg_s, &h->r_ss, &h->r_cost, &h->r_opp,
                      &h->r_nopp, &h->r_key, &h->r_near_i, &h->r_near4};
    for (DevBuf* b : bufs) release(*b);
    for (int i = 0; i < N_PIPE; ++i) {
        PipeSlot& p = h->pipe[i];
        DevBuf* pb[] = {&p.poses, &p.opp, &p.nopp, &p.ctx, &p.centres, &p.best, &p.idx, &p.cost,
                        &p.traj, &p.costs, &p.flags, &p.ss, &p.near_i, &p.near4, &p.prev, &p.pvalid};
        for (DevBuf* b : pb) release(*b);
        if (p.done) cudaEventDestroy(p.done);
        if (p.stream) cudaStreamDestroy(p.stream);
    }
    if (h->gexec) cudaGraphExecDestroy(h->gexec);
    for (int i = 0; i < 4 * F1L_EV_SLOTS; ++i)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    if (h->h_in) cudaFreeHost(h->h_in);
    if (h->h_out) cudaFreeHost(h->h_out);
    if (h->h_detail) cudaFreeHost(h->h_detail);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
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
    static const bool ctab_off = getenv("F1L_CTAB") && atoi(getenv("F1L_CTAB")) == 0;
    if (nblk * 32 <= F1L_CTAB_SEGS && h->device >= 0 && h->device < 64 && !ctab_off) {
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
    release(h->grid);
    release(h->clear);
    release(h->clear_tmp);
    release(h->edt);
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
static int plan_internal(f1l_handle h, const double pose[4], const double* opp, int n_opp,
                         const double* goals, int n_goals, int c_begin, int c_end,
                         int update_prev, f1l_plan_result* out, bool exchange = false,
                         int row0 = 0, int row_step = 1) {
    if (!h || !pose || !out) return F1L_ERR_INVALID_ARG;
    if (n_opp < 0 || n_opp > F1L_MAX_OPP || (n_opp > 0 && !opp)) return F1L_ERR_INVALID_ARG;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    CK(cudaSetDevice(h->device));
    const int C = goals ? n_goals : h->nL * h->nW;
    if (C <= 0) return F1L_ERR_NO_GOALS;
    const int M = h->cfg.n_samples;
    cudaStream_t st = h->stream;

    NvtxRange nvtx_plan("f1l.plan (single query)");
    // stage inputs (pinned)
    QInput* hin = (QInput*)h->h_in;
    memcpy(hin->pose, pose, 4 * sizeof(double));
    hin->n_opp = n_opp;
    hin->pad = 0;
    if (n_opp) memcpy(hin->opp, opp, (size_t)n_opp * 3 * sizeof(double));
    ENS(h->q_in, sizeof(QInput));
    ENS(h->q_ctx, sizeof(QueryCtx));
    ENS(h->q_centres, sizeof(Centre) * (size_t)(h->nL > 0 ? h->nL : 1));
    ENS(h->q_best, 16);   // argmin key | work counter of the persistent-grid schedule
    ENS(h->prev, F1L_MAX_M * sizeof(float));
    // detail block layout (every region 16-byte aligned)
    const size_t c16 = ((size_t)C + 3) & ~(size_t)3;
    const size_t off_costs = 0, off_terms = off_costs + c16 * 4, off_goals = off_terms + c16 * F1L_N_TERMS * 4;
    const size_t off_params = off_goals + c16 * 12, off_flags = off_params + c16 * 16;
    const size_t detail_bytes = off_flags + c16;
    ENS(h->q_detail, detail_bytes);
    const bool want_detail = out->costs || out->terms || out->flags || out->goals || out->params;
    if (want_detail && h->h_detail_cap < detail_bytes) {
        CK(cudaStreamSynchronize(st));
        if (h->h_detail) cudaFreeHost(h->h_detail);
        h->h_detail = nullptr;
        h->h_detail_cap = 0;
        CK(cudaHostAlloc(&h->h_detail, detail_bytes, cudaHostAllocDefault));
        h->h_detail_cap = detail_bytes;
        h->epoch++;   // the captured graph holds the old staging address
    }
    char* ddet = (char*)h->q_detail.p;
    if (out->states) ENS(h->q_states, (size_t)C * M * 16);
    if (out->headings) ENS(h->q_headings, (size_t)C * M * 8);
    const float4* d_goals = nullptr;
    if (goals) {
        std::vector<float> g4(4 * (size_t)C);
        for (int c = 0; c < C; ++c) {
            g4[4 * c] = (float)goals[3 * c];
            g4[4 * c + 1] = (float)goals[3 * c + 1];
            g4[4 * c + 2] = (float)goals[3 * c + 2];
            g4[4 * c + 3] = 0.0f;
        }
        ENS(h->q_goals, (size_t)C * 16);
        CK(cudaMemcpyAsync(h->q_goals.p, g4.data(), (size_t)C * 16, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));  // g4 is a stack-lifetime staging buffer
        d_goals = (const float4*)h->q_goals.p;
    }

    if (!h->q_res.p) {
        ENS(h->q_res, Q_RES_BYTES);
        // the header's padding words travel with the D2H copy: defined bytes (initcheck-clean)
        CK(cudaMemsetAsync(h->q_res.p, 0, sizeof(QHeader), st));
    }
    // Results of a single query: the select kernel writes header and best trajectory straight into
    // the mapped pinned block (posted writes over the host link, 3-10 KB) -- no D2H copy node on the
    // latency path; without a mapping they go to the device block and one D2H copy.
    const bool direct = h->h_out_dev != nullptr;
    char* dres = direct ? (char*)h->h_out_dev : (char*)h->q_res.p;
    BatchOut o;
    o.steer_speed = (double*)(dres + offsetof(QHeader, steer));
    o.best_idx = (int32_t*)(dres + offsetof(QHeader, best_idx));
    o.status = (int32_t*)(dres + offsetof(QHeader, no_feasible));
    o.best_cost = (float*)(dres + offsetof(QHeader, best_cost));
    o.best_traj = (float4*)(dres + Q_OFF_TRAJ);
    o.best_traj_map = out->best_traj_map ? (double*)(dres + Q_OFF_MAP) : nullptr;
    o.costs = (float*)(ddet + off_costs);
    o.terms = out->terms ? (float*)(ddet + off_terms) : nullptr;
    o.flags = out->flags ? (uint8_t*)(ddet + off_flags) : nullptr;
    o.goals_out = out->goals ? (float*)(ddet + off_goals) : nullptr;
    o.params = out->params ? (float4*)(ddet + off_params) : nullptr;
    o.states = out->states ? (float4*)h->q_states.p : nullptr;
    o.headings = out->headings ? (float2*)h->q_headings.p : nullptr;
    o.prev_out = update_prev ? (float*)h->prev.p : nullptr;
    if (row_step > 1) {   // row-interleaved shard: rows row0, row0 + row_step, ... of the goal grid
        if (goals || row0 < 0 || row0 >= row_step) return F1L_ERR_INVALID_ARG;
        const int n_rows = row0 < h->nL ? (h->nL - row0 + row_step - 1) / row_step : 0;
        // More ranks than lookahead rows: with peers attached the call is collective, so a rank
        // without rows must still arrive at the exchange (it contributes key = ~0 and returns the
        // global winner like everybody else); alone there is nothing to answer.
        if (n_rows <= 0) {
            if (!(exchange && h->xview.world > 1)) return F1L_ERR_INVALID_ARG;
            o.empty_shard = true;
        }
        o.row0 = row0;
        o.row_step = row_step;
        c_begin = 0;
        c_end = n_rows * h->nW;
        o.s_row0 = row0 < h->nL ? row0 : 0;   // the sampler fills this shard's rows only
        o.s_step = row_step;
        o.s_rows = n_rows > 0 ? n_rows : 0;
    } else if (!goals && h->nW > 0 && (c_begin > 0 || (c_end > 0 && c_end < C))) {
        // contiguous candidate block: the lookahead rows it touches
        const int cb = c_begin > 0 ? c_begin : 0, ce = (c_end > 0 && c_end < C) ? c_end : C;
        if (cb < ce) {
            o.s_row0 = cb / h->nW;
            o.s_step = 1;
            o.s_rows = (ce - 1) / h->nW - o.s_row0 + 1;
        }
    }
    o.work_next = (int*)((char*)h->q_best.p + 8);
    exchange = exchange && h->xview.world > 1;
    if (exchange) {   // the ranks' minima meet inside select_kernel (peer memory over NVLink)
        o.xc = &h->xview;
        o.xchg_status = (int32_t*)(dres + offsetof(QHeader, pad));
    }
    const bool sharded = exchange || row_step > 1 || c_begin != 0 || (c_end > 0 && c_end < C);
    QHeader* hd = (QHeader*)h->h_out;
    float* htraj = (float*)((char*)h->h_out + sizeof(QHeader));
    const QInput* din = (const QInput*)h->q_in.p;
    // H2D of the input block, the three kernels, D2H of header + best trajectory.  The
    // similarity term reads the previous path while select overwrites it: eval reads it before
    // select runs (stream order), so one buffer suffices.
    auto enqueue = [&](bool time_it) -> int {
        CK(cudaMemcpyAsync(h->q_in.p, hin, sizeof(QInput), cudaMemcpyHostToDevice, st));
        if (sharded && want_detail) {
            // sharded evaluation: untouched candidates keep +inf / zero flags (only when the
            // per-candidate arrays travel back at all)
            fill_f32_kernel<<<(C + 255) / 256, 256, 0, st>>>(o.costs, (size_t)C, INFINITY);
            h->launches += 1;
            if (o.flags) CK(cudaMemsetAsync(o.flags, 0, (size_t)C, st));
        }
        int r = launch_pipeline(h, st, din->pose, din->opp, &din->n_opp, 1, F1L_MAX_OPP, d_goals, C,
                                c_begin, c_end, (QueryCtx*)h->q_ctx.p, (Centre*)h->q_centres.p,
                                (unsigned long long*)h->q_best.p, nullptr, nullptr,
                                h->has_prev ? (const float*)h->prev.p : nullptr, 0, nullptr, o, time_it);
        if (r != F1L_OK) return r;
        if (!direct) {
            CK(cudaMemcpyAsync(hd, h->q_res.p, sizeof(QHeader) + (size_t)M * 16, cudaMemcpyDeviceToHost, st));
            if (o.best_traj_map)
                CK(cudaMemcpyAsync((char*)h->h_out + Q_OFF_MAP, dres + Q_OFF_MAP, (size_t)M * 32,
                                   cudaMemcpyDeviceToHost, st));
        }
        if (want_detail)
            CK(cudaMemcpyAsync(h->h_detail, ddet, detail_bytes, cudaMemcpyDeviceToHost, st));
        return F1L_OK;
    };
    if (h->use_graph && !goals && !h->timing) {
        // the whole chain as one CUDA graph, re-captured only when an upload / config change or
        // the set of requested outputs alters a kernel argument
        const unsigned long long mask = (want_detail ? 256u : 0u) | (out->terms ? 1u : 0u) | (out->flags ? 2u : 0u) |
                                        (out->goals ? 4u : 0u) | (out->params ? 8u : 0u) |
                                        (out->states ? 16u : 0u) | (out->headings ? 32u : 0u) |
                                        (update_prev ? 64u : 0u) | (h->has_prev ? 128u : 0u) |
                                        (exchange ? 512u : 0u) | (out->best_traj_map ? 1024u : 0u);
        // a candidate shard is a constant of the captured kernels too
        const unsigned long long shard_key = ((unsigned long long)(unsigned)c_begin << 32) | (unsigned)c_end;
        const unsigned long long rows_key = ((unsigned long long)(unsigned)row_step << 32) | (unsigned)row0;
        if (!h->gexec || h->gkey[0] != h->epoch || h->gkey[1] != mask || h->gkey[2] != shard_key ||
            h->gkey[3] != rows_key) {
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
            h->gkey[2] = shard_key;
            h->gkey[3] = rows_key;
        }
        CK(cudaGraphLaunch(h->gexec, st));
        h->launches += 3;
    } else {
        int r = enqueue(h->timing != 0);
        if (r != F1L_OK) return r;
    }

    // the big optional arrays go straight into the caller's buffers
    if (out->states) CK(cudaMemcpyAsync(out->states, h->q_states.p, (size_t)C * M * 16, cudaMemcpyDeviceToHost, st));
    if (out->headings) CK(cudaMemcpyAsync(out->headings, h->q_headings.p, (size_t)C * M * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (update_prev) {
        h->has_prev = 1;
        h->prev_m = M;
    }
    if (exchange && hd->pad != 0) return F1L_ERR_PEER_TIMEOUT;
    h->lastq_C = C;
    h->lastq_goals = goals != nullptr;
    h->lastq_rows[0] = o.s_row0;
    h->lastq_rows[1] = o.s_step;
    h->lastq_rows[2] = o.s_rows;
    h->lastq_epoch = h->epoch;
    out->steer = hd->steer;
    out->speed = hd->speed;
    out->best_idx = hd->best_idx;
    out->no_feasible = hd->no_feasible;
    out->tracker_found = hd->tracker_found;
    out->n_candidates = C;
    out->best_cost = hd->best_cost;
    if (out->best_traj) memcpy(out->best_traj, htraj, (size_t)M * 16);
    if (out->best_traj_map) memcpy(out->best_traj_map, (char*)h->h_out + Q_OFF_MAP, (size_t)M * 32);
    if (want_detail) {
        const char* hdet = (const char*)h->h_detail;
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
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, 0, 0, update_prev, out);
}

int f1l_plan_shard(f1l_handle h, const double pose[4], const double* opp, int n_opp, int c_begin,
                   int c_end, f1l_plan_result* out) {
    // with peers attached (f1l_xchg_attach) every rank returns the GLOBAL winner
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, c_begin, c_end, 0, out, true);
}

int f1l_plan_rows(f1l_handle h, const double pose[4], const double* opp, int n_opp, int row_begin,
                  int row_step, int update_prev, f1l_plan_result* out) {
    if (row_step < 1) return F1L_ERR_INVALID_ARG;
    if (row_step == 1) return plan_internal(h, pose, opp, n_opp, nullptr, 0, 0, 0, update_prev, out, true);
    return plan_internal(h, pose, opp, n_opp, nullptr, 0, 0, 0, update_prev, out, true, row_begin, row_step);
}

int f1l_select_candidate(f1l_handle h, int idx, float cost, int update_prev, f1l_plan_result* out) {
    if (!h || !out) return F1L_ERR_INVALID_ARG;
    // the sampler context, goal centres / explicit goals of the last query must still be current
    if (h->lastq_epoch != h->epoch || idx < 0 || idx >= h->lastq_C) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int M = h->cfg.n_samples, C = h->lastq_C;
    unsigned long long* hkey = (unsigned long long*)h->h_in;   // pinned staging
    uint32_t cb;
    memcpy(&cb, &cost, 4);
    const uint32_t ord = (cb & 0x80000000u) ? ~cb : (cb | 0x80000000u);   // float_orderable
    *hkey = ((unsigned long long)ord << 32) | (unsigned)idx;
    CK(cudaMemcpyAsync(h->q_best.p, hkey, 8, cudaMemcpyHostToDevice, st));
    char* dres = (char*)h->q_res.p;
    BatchOut o;
    o.steer_speed = (double*)(dres + offsetof(QHeader, steer));
    o.best_idx = (int32_t*)(dres + offsetof(QHeader, best_idx));
    o.status = (int32_t*)(dres + offsetof(QHeader, no_feasible));
    o.best_cost = (float*)(dres + offsetof(QHeader, best_cost));
    o.best_traj = (float4*)(dres + Q_OFF_TRAJ);
    o.best_traj_map = out->best_traj_map ? (double*)(dres + Q_OFF_MAP) : nullptr;
    o.prev_out = update_prev ? (float*)h->prev.p : nullptr;
    o.s_row0 = h->lastq_rows[0];
    o.s_step = h->lastq_rows[1];
    o.s_rows = h->lastq_rows[2];
    const SelectArgs se = select_args(h, track_view(h), lut_view(h), eval_params(h),
                                      (const QueryCtx*)h->q_ctx.p, (const Centre*)h->q_centres.p,
                                      h->lastq_goals ? (const float4*)h->q_goals.p : nullptr, C, 0,
                                      (const unsigned long long*)h->q_best.p, 1, o);
    eval_bucket_of(M).select<<<1, SELECT_THREADS, 0, st>>>(se);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_out, dres, Q_OFF_TRAJ + (size_t)M * 16, cudaMemcpyDeviceToHost, st));
    if (o.best_traj_map)
        CK(cudaMemcpyAsync((char*)h->h_out + Q_OFF_MAP, dres + Q_OFF_MAP, (size_t)M * 32,
                           cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (update_prev) { h->has_prev = 1; h->prev_m = M; }
    const QHeader* hd = (const QHeader*)h->h_out;
    out->steer = hd->steer;
    out->speed = hd->speed;
    out->best_idx = hd->best_idx;
    out->no_feasible = hd->no_feasible;
    out->tracker_found = hd->tracker_found;
    out->n_candidates = C;
    out->best_cost = hd->best_cost;
    if (out->best_traj) memcpy(out->best_traj, (char*)h->h_out + Q_OFF_TRAJ, (size_t)M * 16);
    if (out->best_traj_map) memcpy(out->best_traj_map, (char*)h->h_out + Q_OFF_MAP, (size_t)M * 32);
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
    return plan_internal(h, pose, opp, n_opp, goals, n_goals, 0, 0, update_prev, out);
}

int f1l_generate(f1l_handle h, const double* goals, int n_goals, float* states, float* params,
                 uint8_t* flags) {
    if (!h || !goals || n_goals <= 0 || !states) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    const int C = n_goals, M = h->cfg.n_samples;
    std::vector<float> g4(4 * (size_t)C);
    for (int c = 0; c < C; ++c) {
        g4[4 * c] = (float)goals[3 * c];
        g4[4 * c + 1] = (float)goals[3 * c + 1];
        g4[4 * c + 2] = (float)goals[3 * c + 2];
        g4[4 * c + 3] = 0.0f;
    }
    ENS(h->q_goals, (size_t)C * 16);
    ENS(h->q_states, (size_t)C * M * 16);
    ENS(h->q_params, (size_t)C * 16);
    ENS(h->q_flags, (size_t)C);
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(h->q_goals.p, g4.data(), (size_t)C * 16, cudaMemcpyHostToDevice, st));
    const int wpc = 8;
    eval_bucket_of(M).generate<<<(C + wpc - 1) / wpc, wpc * 32, 0, st>>>(
        lut_view(h), eval_params(h), (const float4*)h->q_goals.p, C, (float4*)h->q_states.p,
        (float4*)h->q_params.p, (uint8_t*)h->q_flags.p);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(states, h->q_states.p, (size_t)C * M * 16, cudaMemcpyDeviceToHost, st));
    if (params) CK(cudaMemcpyAsync(params, h->q_params.p, (size_t)C * 16, cudaMemcpyDeviceToHost, st));
    if (flags) CK(cudaMemcpyAsync(flags, h->q_flags.p, (size_t)C, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

// ---- batch --------------------------------------------------------------------------------
// prev_theta [S,M] / has_prev [S] (nullable): per-scenario previous paths.  With update_prev the
// select kernel overwrites them in place with each scenario's best trajectory.  That is safe:
// eval_kernel reads a scenario's path in its prologue, and select_kernel writes it in a later
// kernel on the same stream.
static int plan_batch_dev_internal(f1l_handle h, const double* poses_dev, const double* opp_dev,
                                   const int32_t* n_opp_dev, int S, int max_opp, float* prev_theta_dev,
                                   uint8_t* has_prev_dev, int update_prev, int32_t* best_idx_dev,
                                   float* best_cost_dev, float* best_traj_dev, float* costs_dev,
                                   uint8_t* flags_dev, double* steer_speed_dev, void* stream) {
    if (!h || !poses_dev || S <= 0) return F1L_ERR_INVALID_ARG;
    if (max_opp > 0 && !opp_dev) return F1L_ERR_INVALID_ARG;
    if ((update_prev || has_prev_dev) && !prev_theta_dev) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (h->nL * h->nW <= 0) return F1L_ERR_NO_GOALS;
    ENS(h->b_ctx, sizeof(QueryCtx) * (size_t)S);
    ENS(h->b_centres, sizeof(Centre) * (size_t)S * h->nL);
    ENS(h->b_best, 8 * (size_t)S);
    ENS(h->b_near_i, 4 * (size_t)S);
    ENS(h->b_near4, 32 * (size_t)S);
    BatchOut o;
    o.best_idx = best_idx_dev;
    o.best_cost = best_cost_dev;
    o.best_traj = (float4*)best_traj_dev;
    o.costs = costs_dev;
    o.flags = flags_dev;
    o.steer_speed = steer_speed_dev;
    o.prev_out = update_prev ? prev_theta_dev : nullptr;
    o.prev_valid_out = update_prev ? has_prev_dev : nullptr;
    return launch_pipeline(h, (cudaStream_t)stream, poses_dev, max_opp > 0 ? opp_dev : nullptr,
                           n_opp_dev, S, max_opp, nullptr, 0, 0, 0, (QueryCtx*)h->b_ctx.p,
                           (Centre*)h->b_centres.p, (unsigned long long*)h->b_best.p,
                           (int32_t*)h->b_near_i.p, (double*)h->b_near4.p, prev_theta_dev,
                           h->cfg.n_samples, has_prev_dev, o, h->timing != 0);
}

int f1l_plan_batch_dev(f1l_handle h, const double* poses_dev, const double* opp_dev,
                       const int32_t* n_opp_dev, int S, int max_opp, int32_t* best_idx_dev,
                       float* best_cost_dev, float* best_traj_dev, float* costs_dev,
                       uint8_t* flags_dev, double* steer_speed_dev, void* stream) {
    return plan_batch_dev_internal(h, poses_dev, opp_dev, n_opp_dev, S, max_opp, nullptr, nullptr, 0,
                                   best_idx_dev, best_cost_dev, best_traj_dev, costs_dev, flags_dev,
                                   steer_speed_dev, stream);
}

int f1l_plan_batch_prev_dev(f1l_handle h, const double* poses_dev, const double* opp_dev,
                            const int32_t* n_opp_dev, int S, int max_opp, float* prev_theta_dev,
                            uint8_t* has_prev_dev, int update_prev, int32_t* best_idx_dev,
                            float* best_cost_dev, float* best_traj_dev, float* costs_dev,
                            uint8_t* flags_dev, double* steer_speed_dev, void* stream) {
    return plan_batch_dev_internal(h, poses_dev, opp_dev, n_opp_dev, S, max_opp, prev_theta_dev,
                                   has_prev_dev, update_prev, best_idx_dev, best_cost_dev, best_traj_dev,
                                   costs_dev, flags_dev, steer_speed_dev, stream);
}

static int plan_batch_internal(f1l_handle h, const double* poses, const double* opp, const int32_t* n_opp,
                               int S, int max_opp, float* prev_theta, uint8_t* has_prev, int update_prev,
                               int32_t* best_idx, float* best_cost, float* best_traj, float* costs,
                               uint8_t* flags, double* steer_speed) {
    if (!h || !poses || S <= 0) return F1L_ERR_INVALID_ARG;
    if (max_opp > 0 && !opp) return F1L_ERR_INVALID_ARG;
    if ((update_prev || has_prev) && !prev_theta) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    const int C = h->nL * h->nW;
    if (C <= 0) return F1L_ERR_NO_GOALS;
    const int M = h->cfg.n_samples;
    // chunked 3-stream pipeline: H2D(i+1) | kernels(i) | D2H(i-1)
    // 8192-scenario chunks (0.23 M candidates: 1 ms of kernels against ~30 us of launches) for
    // large batches; smaller batches are cut into about eight chunks, down to 1024 scenarios.  The
    // last chunks taper (half, quarter, ... of a chunk, down to 1024): the result copy of the final
    // chunk is the one transfer nothing overlaps, 14 MB at full size but under 2 MB tapered.
    int chunk = 8192;
    bool taper = true;
    if (const char* e = getenv("F1L_PIPE_CHUNK")) { const int v = atoi(e); if (v > 0) { chunk = v; taper = false; } }
    else if (S < 8 * chunk) { chunk = (S + 7) / 8; if (chunk < 1024) chunk = 1024; }
    if (chunk > S) chunk = S;
    int slot = 0;
    for (int s0 = 0, n = 0; s0 < S; s0 += n, slot = (slot + 1) % N_PIPE) {
        n = (S - s0 < chunk) ? (S - s0) : chunk;
        if (taper) {
            // rest = what is left after this chunk: keep halving while the tail is short
            const int rest = S - s0;
            if (rest < 2 * chunk && rest > 1024) { n = rest / 2; if (n < 1024) n = 1024; if (n > rest) n = rest; }
        }
        NvtxRange nvtx_chunk("f1l.plan_batch.chunk (H2D, kernels, D2H)");
        PipeSlot& p = h->pipe[slot];
        cudaStream_t st = p.stream;
        CK(cudaStreamSynchronize(st));  // slot buffers free again (grow-only ensure below)
        ENS(p.poses, (size_t)n * 32);
        if (max_opp > 0) ENS(p.opp, (size_t)n * max_opp * 24);
        if (n_opp) ENS(p.nopp, (size_t)n * 4);
        ENS(p.ctx, sizeof(QueryCtx) * (size_t)n);
        ENS(p.centres, sizeof(Centre) * (size_t)n * h->nL);
        ENS(p.best, 8 * (size_t)n);
        ENS(p.near_i, 4 * (size_t)n);
        ENS(p.near4, 32 * (size_t)n);
        if (best_idx) ENS(p.idx, (size_t)n * 4);
        if (best_cost) ENS(p.cost, (size_t)n * 4);
        if (best_traj) ENS(p.traj, (size_t)n * M * 16);
        if (costs) ENS(p.costs, (size_t)n * C * 4);
        if (flags) ENS(p.flags, (size_t)n * C);
        if (steer_speed) ENS(p.ss, (size_t)n * 16);
        if (prev_theta) ENS(p.prev, (size_t)n * M * 4);
        if (has_prev) ENS(p.pvalid, (size_t)n);
        CK(cudaMemcpyAsync(p.poses.p, poses + 4 * (size_t)s0, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        if (max_opp > 0)
            CK(cudaMemcpyAsync(p.opp.p, opp + 3 * (size_t)max_opp * s0, (size_t)n * max_opp * 24,
                               cudaMemcpyHostToDevice, st));
        if (n_opp) CK(cudaMemcpyAsync(p.nopp.p, n_opp + s0, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        if (prev_theta)
            CK(cudaMemcpyAsync(p.prev.p, prev_theta + (size_t)M * s0, (size_t)n * M * 4, cudaMemcpyHostToDevice, st));
        if (has_prev) CK(cudaMemcpyAsync(p.pvalid.p, has_prev + s0, (size_t)n, cudaMemcpyHostToDevice, st));
        BatchOut o;
        o.best_idx = best_idx ? (int32_t*)p.idx.p : nullptr;
        o.best_cost = best_cost ? (float*)p.cost.p : nullptr;
        o.best_traj = best_traj ? (float4*)p.traj.p : nullptr;
        o.costs = costs ? (float*)p.costs.p : nullptr;
        o.flags = flags ? (uint8_t*)p.flags.p : nullptr;
        o.steer_speed = steer_speed ? (double*)p.ss.p : nullptr;
        // in place on the slot's copies, as in plan_batch_dev_internal
        o.prev_out = update_prev ? (float*)p.prev.p : nullptr;
        o.prev_valid_out = update_prev && has_prev ? (uint8_t*)p.pvalid.p : nullptr;
        int r = launch_pipeline(h, st, (const double*)p.poses.p,
                                max_opp > 0 ? (const double*)p.opp.p : nullptr,
                                n_opp ? (const int32_t*)p.nopp.p : nullptr, n, max_opp, nullptr, 0,
                                0, 0, (QueryCtx*)p.ctx.p, (Centre*)p.centres.p,
                                (unsigned long long*)p.best.p, (int32_t*)p.near_i.p,
                                (double*)p.near4.p, prev_theta ? (const float*)p.prev.p : nullptr, M,
                                has_prev ? (const uint8_t*)p.pvalid.p : nullptr, o, false);
        if (r != F1L_OK) return r;
        if (best_idx) CK(cudaMemcpyAsync(best_idx + s0, p.idx.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        if (best_cost) CK(cudaMemcpyAsync(best_cost + s0, p.cost.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        if (best_traj)
            CK(cudaMemcpyAsync(best_traj + 4 * (size_t)M * s0, p.traj.p, (size_t)n * M * 16,
                               cudaMemcpyDeviceToHost, st));
        if (costs) CK(cudaMemcpyAsync(costs + (size_t)C * s0, p.costs.p, (size_t)n * C * 4, cudaMemcpyDeviceToHost, st));
        if (flags) CK(cudaMemcpyAsync(flags + (size_t)C * s0, p.flags.p, (size_t)n * C, cudaMemcpyDeviceToHost, st));
        if (steer_speed) CK(cudaMemcpyAsync(steer_speed + 2 * (size_t)s0, p.ss.p, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
        if (update_prev) {
            CK(cudaMemcpyAsync(prev_theta + (size_t)M * s0, p.prev.p, (size_t)n * M * 4, cudaMemcpyDeviceToHost, st));
            if (has_prev) CK(cudaMemcpyAsync(has_prev + s0, p.pvalid.p, (size_t)n, cudaMemcpyDeviceToHost, st));
        }
    }
    for (int i = 0; i < N_PIPE; ++i) CK(cudaStreamSynchronize(h->pipe[i].stream));
    return F1L_OK;
}

int f1l_plan_batch(f1l_handle h, const double* poses, const double* opp, const int32_t* n_opp,
                   int S, int max_opp, int32_t* best_idx, float* best_cost, float* best_traj,
                   float* costs, uint8_t* flags, double* steer_speed) {
    return plan_batch_internal(h, poses, opp, n_opp, S, max_opp, nullptr, nullptr, 0, best_idx, best_cost,
                               best_traj, costs, flags, steer_speed);
}

int f1l_plan_batch_prev(f1l_handle h, const double* poses, const double* opp, const int32_t* n_opp,
                        int S, int max_opp, float* prev_theta, uint8_t* has_prev, int update_prev,
                        int32_t* best_idx, float* best_cost, float* best_traj, float* costs,
                        uint8_t* flags, double* steer_speed) {
    return plan_batch_internal(h, poses, opp, n_opp, S, max_opp, prev_theta, has_prev, update_prev, best_idx,
                               best_cost, best_traj, costs, flags, steer_speed);
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

int f1l_rollout_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_fleet* fl, int S,
                    int n_steps, const f1l_rollout_trace* trace, void* stream) {
    if (!h || !rc || !fl) return F1L_ERR_INVALID_ARG;
    if (!fl->state || !fl->prev_theta || !fl->has_prev || !fl->status || !fl->progress ||
        !fl->track_i || !fl->track_s)
        return F1L_ERR_INVALID_ARG;
    if (rc->group < 1 || rc->group > F1L_MAX_GROUP || S <= 0 || S % rc->group != 0) return F1L_ERR_INVALID_ARG;
    if (rc->substeps < 1 || n_steps < 0) return F1L_ERR_INVALID_ARG;
    if (!(rc->dt > 0) || !(rc->max_steer > 0) || !(rc->max_accel > 0) || !(rc->v_max > 0))
        return F1L_ERR_INVALID_ARG;
    if (n_steps == 0) return F1L_OK;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    if (h->nL * h->nW <= 0) return F1L_ERR_NO_GOALS;
    CK(cudaSetDevice(h->device));
    ENS(h->r_ss, (size_t)S * 16);
    ENS(h->r_cost, (size_t)S * 4);
    ENS(h->r_opp, (size_t)S * F1L_MAX_OPP * 24);
    ENS(h->r_nopp, (size_t)S * 4);
    ENS(h->r_key, (size_t)S * 8);
    ENS(h->r_near_i, (size_t)S * 4);
    ENS(h->r_near4, (size_t)S * 32);
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
    const unsigned blocks = (unsigned)((a.n_races + ROLLOUT_WARPS - 1) / ROLLOUT_WARPS);

    // once per call: global nearest_point of every car (K1) for the cars to re-acquire, then the
    // initial pass of the step kernel (no integration) builds step 0's opponent table
    PPOut po;
    memset(&po, 0, sizeof(po));
    po.nearest = (double*)h->r_near4.p;
    po.nearest_i = (int32_t*)h->r_near_i.p;
    launch_pp(a.tr, st, fl->state, 4, S, -1.0, h->cfg.wheelbase, 0.0, 0, 0.0,
              (unsigned long long*)h->r_key.p, pp_slots(h), po, ctab_valid(h), h);
    a.near_i = po.nearest_i;
    a.near4 = po.nearest;
    rollout_step_kernel<<<blocks, ROLLOUT_WARPS * 32, 0, st>>>(a);
    h->launches += 3;
    CK(cudaGetLastError());
    a.near_i = nullptr;
    a.near4 = nullptr;
    a.steer_speed = (const double*)h->r_ss.p;
    a.best_cost = (const float*)h->r_cost.p;
    for (int k = 0; k < n_steps; ++k) {
        const size_t row = (size_t)k * S;
        int32_t* best_idx = trace && trace->best_idx ? trace->best_idx + row : nullptr;
        const int r = plan_batch_dev_internal(h, fl->state, a.opp, a.n_opp, S, F1L_MAX_OPP, fl->prev_theta,
                                              fl->has_prev, 1, best_idx, (float*)h->r_cost.p, nullptr,
                                              nullptr, nullptr, (double*)h->r_ss.p, stream);
        if (r != F1L_OK) return r;
        a.tr_state = trace && trace->state ? trace->state + 4 * row : nullptr;
        a.tr_ss = trace && trace->steer_speed ? trace->steer_speed + 2 * row : nullptr;
        a.tr_status = trace && trace->status ? trace->status + row : nullptr;
        a.tr_progress = trace && trace->progress ? trace->progress + row : nullptr;
        rollout_step_kernel<<<blocks, ROLLOUT_WARPS * 32, 0, st>>>(a);
        h->launches += 1;
        CK(cudaGetLastError());
    }
    return F1L_OK;
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
    PPOut o;
    o.nearest = nearest_dev;
    o.nearest_i = nearest_i_dev;
    o.lookahead = lookahead_dev;
    o.lookahead_i = lookahead_i_dev;
    o.actuation = actuation_dev;
    o.status = status_dev;
    o.front = nullptr;
    ENS(h->pp_key, (size_t)n_poses * 8);   // scan scratch (one call in flight per handle)
    launch_pp(track_view(h), (cudaStream_t)stream, poses_dev, 3, n_poses, L, h->cfg.wheelbase,
              h->cfg.max_reacquire, 0, 0.0, (unsigned long long*)h->pp_key.p, pp_slots(h), o, ctab_valid(h), h);
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
    ENS(h->m_in, (size_t)n * 24);
    if (nearest) ENS(h->m_o0, (size_t)n * 32);
    if (nearest_i) ENS(h->m_o1, (size_t)n * 4);
    if (lookahead) ENS(h->m_o2, (size_t)n * 32);
    if (lookahead_i) ENS(h->m_o3, (size_t)n * 4);
    if (actuation) ENS(h->m_o4, (size_t)n * 16);
    if (status) ENS(h->m_o5, (size_t)n * 4);
    CK(cudaMemcpyAsync(h->m_in.p, poses, (size_t)n * 24, cudaMemcpyHostToDevice, st));
    int r = f1l_pure_pursuit_batch_dev(
        h, (const double*)h->m_in.p, n, L, nearest ? (double*)h->m_o0.p : nullptr,
        nearest_i ? (int32_t*)h->m_o1.p : nullptr, lookahead ? (double*)h->m_o2.p : nullptr,
        lookahead_i ? (int32_t*)h->m_o3.p : nullptr, actuation ? (double*)h->m_o4.p : nullptr,
        status ? (int32_t*)h->m_o5.p : nullptr, st);
    if (r != F1L_OK) return r;
    if (nearest) CK(cudaMemcpyAsync(nearest, h->m_o0.p, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
    if (nearest_i) CK(cudaMemcpyAsync(nearest_i, h->m_o1.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (lookahead) CK(cudaMemcpyAsync(lookahead, h->m_o2.p, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
    if (lookahead_i) CK(cudaMemcpyAsync(lookahead_i, h->m_o3.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (actuation) CK(cudaMemcpyAsync(actuation, h->m_o4.p, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
    if (status) CK(cudaMemcpyAsync(status, h->m_o5.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

int f1l_front_axle_batch_dev(f1l_handle h, const double* poses_dev, int n_poses, double wheelbase,
                             double k_path, double* front_dev, int32_t* nearest_i_dev,
                             void* stream) {
    if (!h || !poses_dev || n_poses <= 0 || !front_dev) return F1L_ERR_INVALID_ARG;
    if (h->n < 2) return F1L_ERR_NO_TRACK;
    CK(cudaSetDevice(h->device));
    PPOut o;
    o.nearest = nullptr;
    o.nearest_i = nearest_i_dev;
    o.lookahead = nullptr;
    o.lookahead_i = nullptr;
    o.actuation = nullptr;
    o.status = nullptr;
    o.front = front_dev;
    ENS(h->pp_key, (size_t)n_poses * 8);
    launch_pp(track_view(h), (cudaStream_t)stream, poses_dev, 4, n_poses, 0.0, wheelbase, 0.0, 1,
              k_path, (unsigned long long*)h->pp_key.p, pp_slots(h), o, ctab_valid(h), h);
    h->launches += 2;
    CK(cudaGetLastError());
    return F1L_OK;
}

int f1l_front_axle_batch(f1l_handle h, const double* poses, int n, double wheelbase, double k_path,
                         double* front, int32_t* nearest_i) {
    if (!h || !poses || n <= 0 || !front) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    ENS(h->m_in, (size_t)n * 32);
    ENS(h->m_o0, (size_t)n * 48);
    if (nearest_i) ENS(h->m_o1, (size_t)n * 4);
    CK(cudaMemcpyAsync(h->m_in.p, poses, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    int r = f1l_front_axle_batch_dev(h, (const double*)h->m_in.p, n, wheelbase, k_path,
                                     (double*)h->m_o0.p, nearest_i ? (int32_t*)h->m_o1.p : nullptr, st);
    if (r != F1L_OK) return r;
    CK(cudaMemcpyAsync(front, h->m_o0.p, (size_t)n * 48, cudaMemcpyDeviceToHost, st));
    if (nearest_i) CK(cudaMemcpyAsync(nearest_i, h->m_o1.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
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
    ENS(h->m_in, (size_t)n * 16);
    ENS(h->m_in2, (size_t)n * 8);
    ENS(h->m_o0, (size_t)n * 32);
    ENS(h->m_o1, (size_t)n * 4);
    CK(cudaMemcpyAsync(h->m_in.p, points, (size_t)n * 16, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->m_in2.p, t_start, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    intersect_batch_kernel<<<(n + 63) / 64, 64, 0, st>>>(
        track_view(h), (const double*)h->m_in.p, (const double*)h->m_in2.p, n, radius, wrap,
        (double*)h->m_o0.p, (int32_t*)h->m_o1.p);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, h->m_o0.p, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_i, h->m_o1.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

int f1l_get_actuation_batch(f1l_handle h, const double* in, int n, double wheelbase, double* out) {
    if (!h || !in || n <= 0 || !out) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    ENS(h->m_in, (size_t)n * 56);
    ENS(h->m_o0, (size_t)n * 16);
    CK(cudaMemcpyAsync(h->m_in.p, in, (size_t)n * 56, cudaMemcpyHostToDevice, st));
    actuation_batch_kernel<<<(n + 63) / 64, 64, 0, st>>>((const double*)h->m_in.p, n, wheelbase,
                                                         (double*)h->m_o0.p);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, h->m_o0.p, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return F1L_OK;
}

// debug: the last single query's context (teacher-forced collision tests):
// out[0..1] cos/sin pose, [2..7] grid A00 A01 A10 A11 fx fy, [8..9] gix giy (as float bits via
// int copy), [10..] opponents 16 x (x, y, cos, sin)
int f1l_debug_query_ctx(f1l_handle h, float* out_f, int32_t* out_i) {
    if (!h || !out_f || !out_i || !h->q_ctx.p) return F1L_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    QueryCtx q;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(&q, h->q_ctx.p, sizeof(q), cudaMemcpyDeviceToHost));
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
    ENS(h->m_o0, (size_t)h->sm_count * 8 * 256 * 4);
    cudaStream_t st = h->stream;
    const int blocks = h->sm_count * 8, threads = 256, iters = 4096;
    float ms = 0.f;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        ffma_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m_o0.p, iters, 1.0001f, 0.5f);
        CK(cudaEventRecord(h->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    }
    h->launches += 3;
    if (fp32_tflops)
        *fp32_tflops = 2.0 * PEAK_CHAINS * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        mufu_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m_o0.p, iters);
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
        ffma2_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m_o0.p, iters, 1.0001f, 0.5f);
        CK(cudaEventRecord(h->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    }
    out[2] = 4.0 * PEAK_CHAINS * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(h->ev[0], st));
        mixed_peak_kernel<<<blocks, threads, 0, st>>>((float*)h->m_o0.p, iters, 1.0001f, 0.5f);
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
