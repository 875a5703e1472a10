// f1l_lattice.cuh -- K2 sampler, K3+K4 fused spiral generation / cost / collision, K5 select.
//
// One warp per candidate.  FP32 FMA + MUFU math; float64 only where the reference's own float64
// functions are being reproduced (sampler nearest/intersect, tracker).
//
//   sample_kernel  : per scenario -- nearest_point on the raceline, one intersect_point per
//                    lookahead row, goal centres, ego-frame opponents, grid transform, window.
//                    (intent of lattice_planner.py:223-260, SURVEY B.1)
//   eval_kernel    : per candidate -- LUT seed, I Newton steps on (p1, p2, s_f) with a 32-node
//                    Simpson rule (one node per lane), M arc samples by per-interval Simpson and
//                    a warp scan, cost terms (lattice_planner.py:268-296 + raceline deviation
//                    with nearest_point semantics, utils.py:37-67), rectangle-vs-opponent SAT and
//                    occupancy-grid probes, packed 64-bit atomicMin argmin
//                    (lattice_planner.py:159-172).
//   select_kernel  : per scenario -- decode the argmin, regenerate the winning trajectory, run
//                    the pure-pursuit tracker on it (lattice_planner.py:204-214).
#pragma once
#include "f1l_common.cuh"

// ---------------------------------------------------------------------------------------------
// cubic spiral, FP32 (SURVEY B.2 / B.3)
// ---------------------------------------------------------------------------------------------
struct SpiralF {
    float p0, p3;
    float p1, p2, sf;
    float h1, h2, h3;  // b1/2, b2/3, b3/4   (theta polynomial)
    float b1, b2, b3;  // curvature polynomial
};

__device__ __forceinline__ void spiral_set(SpiralF& s) {
    s.b1 = 0.5f * (-11.0f * s.p0 + 18.0f * s.p1 - 9.0f * s.p2 + 2.0f * s.p3);
    s.b2 = 0.5f * (18.0f * s.p0 - 45.0f * s.p1 + 36.0f * s.p2 - 9.0f * s.p3);
    s.b3 = 0.5f * (-9.0f * s.p0 + 27.0f * s.p1 - 27.0f * s.p2 + 9.0f * s.p3);
    s.h1 = 0.5f * s.b1;
    s.h2 = (1.0f / 3.0f) * s.b2;
    s.h3 = 0.25f * s.b3;
}
__device__ __forceinline__ float spiral_g(const SpiralF& s, float u) {
    return u * fmaf(u, fmaf(u, fmaf(u, s.h3, s.h2), s.h1), s.p0);
}
__device__ __forceinline__ float spiral_kappa(const SpiralF& s, float u) {
    return fmaf(u, fmaf(u, fmaf(u, s.b3, s.b2), s.b1), s.p0);
}

// all-reduce (sum) of 8 values per lane over each 8-lane group with 7 + 8 shuffles instead of 24:
// three halving steps leave each lane with one column total, then 8 broadcasts in the group.
__device__ __forceinline__ void group8_allreduce8(float (&v)[8], int lane) {
    const bool h4 = lane & 4, h2 = lane & 2, h1 = lane & 1;
    float a[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float keep = h4 ? v[j + 4] : v[j];
        const float send = h4 ? v[j] : v[j + 4];
        a[j] = keep + __shfl_xor_sync(F1L_FULL, send, 4);
    }
    float b[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float keep = h2 ? a[j + 2] : a[j];
        const float send = h2 ? a[j] : a[j + 2];
        b[j] = keep + __shfl_xor_sync(F1L_FULL, send, 2);
    }
    const float keep = h1 ? b[1] : b[0];
    const float send = h1 ? b[0] : b[1];
    const float c = keep + __shfl_xor_sync(F1L_FULL, send, 1);
    // lane l of a group now holds the total of column l & 7
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __shfl_sync(F1L_FULL, c, j, 8);
}

// Up to `iters` Newton steps q <- q - J^-1 r on FOUR candidates per warp: each 8-lane group owns
// one candidate (its lanes hold the same goal and iterate), each lane four consecutive Simpson
// nodes (lane & 7) * 4 + m + 1 of 32 (node 0 is analytic: cos 0 = 1 and every other integrand
// vanishes there).  A quadrature pass costs about the same instructions as one candidate on 32
// lanes did, but serves four.  A group leaves when its residual reaches the FP32 noise floor, or
// right after a step taken from a residual small enough that the step itself reaches it
// (Newton is quadratic); the warp leaves when all groups have, so a LUT-seeded candidate
// typically spends 2-3 passes, not `iters`.  Callers with one candidate give all groups the
// same goal (same arithmetic, hence bit-identical parameters, as a batch).  `active` = this
// group has a candidate.  Returns the number of quadrature passes this group used.
__device__ __forceinline__ int spiral_newton_g8(SpiralF& sp, float gx, float gy, float gth,
                                                int iters, int lane, bool active) {
    const int l8 = lane & 7;
    float u[4], w[4], d1[4], d2[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        const int j = l8 * 4 + m + 1;
        u[m] = (float)j * (1.0f / 32.0f);
        w[m] = (j == 32) ? (1.0f / 96.0f) : ((j & 1) ? (4.0f / 96.0f) : (2.0f / 96.0f));
        const float u2 = u[m] * u[m];
        d1[m] = u2 * fmaf(u[m], fmaf(u[m], 3.375f, -7.5f), 4.5f);
        d2[m] = u2 * fmaf(u[m], fmaf(u[m], -3.375f, 6.0f), -2.25f);
    }
    const float gmax = fmaxf(1.0f, fmaxf(fabsf(gx), fmaxf(fabsf(gy), fabsf(gth))));
    const float eps = 1.5e-6f * gmax;
    const float eps_step = 2e-4f * gmax;
    bool done = !active;
    int it = 0;
    for (int pass = 0; pass < iters; ++pass) {
        if (__all_sync(F1L_FULL, done)) break;
        spiral_set(sp);
        float v[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const float g = spiral_g(sp, u[m]);
            float s, c;
            __sincosf(sp.sf * g, &s, &c);
            const float wc = w[m] * c, ws = w[m] * s;
            v[0] += wc; v[1] += ws;
            v[2] = fmaf(wc, g, v[2]); v[3] = fmaf(ws, g, v[3]);
            v[4] = fmaf(wc, d1[m], v[4]); v[5] = fmaf(ws, d1[m], v[5]);
            v[6] = fmaf(wc, d2[m], v[6]); v[7] = fmaf(ws, d2[m], v[7]);
        }
        group8_allreduce8(v, lane);
        const float C0 = v[0] + (1.0f / 96.0f), S0 = v[1], Cg = v[2], Sg = v[3];
        const float C1 = v[4], S1 = v[5], C2 = v[6], S2 = v[7];
        const float sf = sp.sf, sf2 = sf * sf;
        const float g1 = 0.125f * (sp.p0 + 3.0f * sp.p1 + 3.0f * sp.p2 + sp.p3);
        const float r0 = fmaf(sf, C0, -gx), r1 = fmaf(sf, S0, -gy), r2 = fmaf(sf, g1, -gth);
        const float rmax = fmaxf(fabsf(r0), fmaxf(fabsf(r1), fabsf(r2)));
        if (!done) {
            ++it;
            if (rmax < eps) {
                done = true;
            } else {
                const float J00 = -sf2 * S1, J01 = -sf2 * S2, J02 = fmaf(-sf, Sg, C0);
                const float J10 = sf2 * C1, J11 = sf2 * C2, J12 = fmaf(sf, Cg, S0);
                const float J20 = 0.375f * sf, J21 = J20, J22 = g1;
                const float m0 = J11 * J22 - J12 * J21, m1 = J10 * J22 - J12 * J20, m2 = J10 * J21 - J11 * J20;
                const float det = J00 * m0 - J01 * m1 + J02 * m2;
                const float inv = __fdividef(1.0f, det);
                const float n0 = r1 * J22 - J12 * r2, n1 = r1 * J21 - J11 * r2, n2 = J10 * r2 - r1 * J20;
                sp.p1 -= (r0 * m0 - J01 * n0 + J02 * n1) * inv;
                sp.p2 -= (J00 * n0 - r0 * m1 + J02 * n2) * inv;
                sp.sf -= (-J00 * n1 - J01 * n2 + r0 * m2) * inv;
                if (rmax < eps_step) done = true;
            }
        }
    }
    spiral_set(sp);
    return it;
}

// nearest-cell LUT seed (the seed the oracle starts from)
__device__ __forceinline__ float4 lut_lookup(const LutView& lut, float gx, float gy, float gth) {
    int ix = __float2int_rd(fmaf(gx - lut.x0, lut.sx, 0.5f));
    int iy = __float2int_rd(fmaf(gy - lut.y0, lut.sy, 0.5f));
    int it = __float2int_rd(fmaf(gth - lut.t0, lut.st, 0.5f));
    ix = min(max(ix, 0), lut.nx - 1);
    iy = min(max(iy, 0), lut.ny - 1);
    it = min(max(it, 0), lut.nt - 1);
    return __ldg(lut.cells + ((size_t)ix * lut.ny + iy) * lut.nt + it);
}

// Trilinear LUT seed per 8-lane group: lane & 7 owns one corner of the goal's cell, three xor
// steps sum the weighted corners on every lane of the group.  The converged cells are samples of
// one smooth solution family, so the interpolated seed lies in the same Newton basin as the nearest
// cell (the oracle's seed) but an order closer to the root: one quadrature pass fewer.  Goals
// outside the table or next to a non-converged cell take the nearest cell.  Branch-free: the four
// groups of a warp may hold different goals.
__device__ __forceinline__ float4 lut_seed(const LutView& lut, float gx, float gy, float gth,
                                           int lane) {
    const float fx = (gx - lut.x0) * lut.sx, fy = (gy - lut.y0) * lut.sy, ft = (gth - lut.t0) * lut.st;
    const bool inside = lut.nx > 1 && lut.ny > 1 && lut.nt > 1 && fx >= 0.0f && fy >= 0.0f &&
                        ft >= 0.0f && fx <= (float)(lut.nx - 1) && fy <= (float)(lut.ny - 1) &&
                        ft <= (float)(lut.nt - 1);
    const int ix = max(min(__float2int_rd(fx), lut.nx - 2), 0), iy = max(min(__float2int_rd(fy), lut.ny - 2), 0);
    const int it = max(min(__float2int_rd(ft), lut.nt - 2), 0);
    const float wx = fx - (float)ix, wy = fy - (float)iy, wt = ft - (float)it;
    const int cx = lane & 1, cy = (lane >> 1) & 1, ct = (lane >> 2) & 1;
    const int jx = min(ix + cx, lut.nx - 1), jy = min(iy + cy, lut.ny - 1), jt = min(it + ct, lut.nt - 1);
    const float4 cell = __ldg(lut.cells + ((size_t)jx * lut.ny + jy) * lut.nt + jt);
    const float w = (cx ? wx : 1.0f - wx) * (cy ? wy : 1.0f - wy) * (ct ? wt : 1.0f - wt);
    float a = w * cell.x, b = w * cell.y, c = w * cell.z;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        a += __shfl_xor_sync(F1L_FULL, a, o);
        b += __shfl_xor_sync(F1L_FULL, b, o);
        c += __shfl_xor_sync(F1L_FULL, c, o);
    }
    const unsigned conv = __ballot_sync(F1L_FULL, cell.w != 0.0f);
    const bool ok = inside && ((conv >> (lane & 24)) & 0xffu) == 0xffu;
    const float4 nearest = lut_lookup(lut, gx, gy, gth);
    return ok ? make_float4(a, b, c, 1.0f) : nearest;
}

// G1 Hermite clothoid from (0,0,0) to the goal -- the generator the reference calls
// (Clothoid.G1Hermite, lattice_planner.py:196); Bertolazzi & Frego 2015.  With the chord as x
// axis: phi0 = -phi, phi1 = gth - phi, delta = phi1 - phi0; 1-D Newton on
//   g(A) = int_0^1 sin(A t^2 + (delta - A) t + phi0) dt = 0      from A = 3 (phi0 + phi1),
// then L = r / int cos, kappa0 = (delta - A)/L, dkappa = 2A/L^2.  Lane = Simpson node
// (lane+1)/32; node 0 contributes sin/cos(phi0)/96 to g and X and nothing to g'.  The clothoid
// is the cubic spiral with linear curvature, so the result is returned as a SpiralF and shares
// the sampling / cost / collision code.  Returns the number of quadrature passes.
__device__ __forceinline__ float wrap_pi_f(float a) {
    const float two_pi = 6.283185307179586f, pi = 3.14159265358979f;
    a -= two_pi * rintf(a * (1.0f / two_pi));
    if (a <= -pi) a += two_pi;
    if (a > pi) a -= two_pi;
    return a;
}

__device__ __forceinline__ int clothoid_g1(SpiralF& sp, float gx, float gy, float gth, int iters,
                                           int lane) {
    const float r = sqrtf(fmaf(gx, gx, gy * gy));
    const float phi = atan2f(gy, gx);
    const float phi0 = wrap_pi_f(-phi), phi1 = wrap_pi_f(gth - phi);
    const float delta = phi1 - phi0;
    const float t = (float)(lane + 1) * (1.0f / 32.0f);
    const float w = (lane == 31) ? (1.0f / 96.0f) : (((lane + 1) & 1) ? (4.0f / 96.0f) : (2.0f / 96.0f));
    const float tt = t * t, dt = tt - t;
    float s0, c0;
    __sincosf(phi0, &s0, &c0);
    float A = 3.0f * (phi0 + phi1), X = 1.0f;
    int it = 0;
    for (;; ++it) {
        float sn, cs;
        __sincosf(fmaf(A, tt, fmaf(delta - A, t, phi0)), &sn, &cs);
        float g = w * sn, x = w * cs, dg = x * dt;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            g += __shfl_xor_sync(F1L_FULL, g, o);
            x += __shfl_xor_sync(F1L_FULL, x, o);
            dg += __shfl_xor_sync(F1L_FULL, dg, o);
        }
        g = fmaf(s0, 1.0f / 96.0f, g);
        X = fmaf(c0, 1.0f / 96.0f, x);
        if (fabsf(g) < 1.5e-6f || it >= iters) { ++it; break; }
        A -= __fdividef(g, dg);
    }
    const float L = __fdividef(r, X);
    sp.sf = L;
    sp.p0 = __fdividef(delta - A, L);          // kappa0
    sp.b1 = 2.0f * A * __fdividef(1.0f, L);    // dkappa * L
    sp.b2 = 0.0f; sp.b3 = 0.0f;
    sp.h1 = 0.5f * sp.b1; sp.h2 = 0.0f; sp.h3 = 0.0f;
    sp.p1 = sp.p0 + sp.b1 * (1.0f / 3.0f);
    sp.p2 = sp.p0 + sp.b1 * (2.0f / 3.0f);
    sp.p3 = sp.p0 + sp.b1;
    return it;
}

// Cubic-spiral generator for the candidate of this lane's 8-lane group (`active`: the group has
// one): LUT seed + Newton.  Returns the quadrature passes the group used.
__device__ __forceinline__ int generate_cubic_g8(SpiralF& sp, const LutView& lut, const EvalParams& ep,
                                                 float gx, float gy, float gth, float p3, int lane,
                                                 bool active) {
    sp.p0 = 0.0f;
    sp.p3 = p3;
    const float4 seed = lut_seed(lut, gx, gy, gth, lane);
    sp.p1 = seed.x; sp.p2 = seed.y; sp.sf = seed.z;
    return spiral_newton_g8(sp, gx, gy, gth, ep.n_newton, lane, active);
}

// generator dispatch for ONE candidate on the whole warp (warp-uniform arguments): fills `sp` for
// the goal, returns the quadrature passes
__device__ __forceinline__ int generate_spiral(SpiralF& sp, const LutView& lut, const EvalParams& ep,
                                               float gx, float gy, float gth, float p3, int lane) {
    if (ep.generator == 1) return clothoid_g1(sp, gx, gy, gth, ep.n_newton, lane);
    return generate_cubic_g8(sp, lut, ep, gx, gy, gth, p3, lane, true);
}

// M arc samples, lane l owns samples [l*IPL, (l+1)*IPL).  Per-interval Simpson
// dx_i = h/6 (cos th_{i-1} + 4 cos th_{i-1/2} + cos th_i), inclusive prefix by a warp scan.
template <int IPL>
__device__ __forceinline__ void spiral_sample(const SpiralF& sp, int M, int lane, float (&x)[IPL],
                                              float (&y)[IPL], float (&th)[IPL], float (&kp)[IPL],
                                              float (&cs)[IPL], float (&sn)[IPL]) {
    const float inv = 1.0f / (float)(M - 1);
    const float h6 = sp.sf * inv * (1.0f / 6.0f);
    const int i0 = lane * IPL;
#pragma unroll
    for (int j = 0; j < IPL; ++j) {
        const float u = (float)(i0 + j) * inv;
        th[j] = sp.sf * spiral_g(sp, u);
        kp[j] = spiral_kappa(sp, u);
        __sincosf(th[j], &sn[j], &cs[j]);
    }
    // cos/sin at the node before this lane's first sample
    float cprev = __shfl_up_sync(F1L_FULL, cs[IPL - 1], 1);
    float sprev = __shfl_up_sync(F1L_FULL, sn[IPL - 1], 1);
    float accx = 0.0f, accy = 0.0f;
#pragma unroll
    for (int j = 0; j < IPL; ++j) {
        const int i = i0 + j;
        const float um = ((float)i - 0.5f) * inv;
        float sm, cm;
        __sincosf(sp.sf * spiral_g(sp, um), &sm, &cm);
        float dx = h6 * (cprev + 4.0f * cm + cs[j]);
        float dy = h6 * (sprev + 4.0f * sm + sn[j]);
        if (i == 0 || i >= M) { dx = 0.0f; dy = 0.0f; }
        accx += dx;
        accy += dy;
        x[j] = accx;
        y[j] = accy;
        cprev = cs[j];
        sprev = sn[j];
    }
    // exclusive scan of the lane totals
    float ix = accx, iy = accy;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float nx = __shfl_up_sync(F1L_FULL, ix, o);
        const float ny = __shfl_up_sync(F1L_FULL, iy, o);
        if (lane >= o) { ix += nx; iy += ny; }
    }
    const float ox = ix - accx, oy = iy - accy;
#pragma unroll
    for (int j = 0; j < IPL; ++j) { x[j] += ox; y[j] += oy; }
}

// ---------------------------------------------------------------------------------------------
// kernel arguments
// ---------------------------------------------------------------------------------------------
struct SampleArgs {
    TrackView tr;
    GridView grid;
    EvalParams ep;
    const double* poses;     // [S,4]
    const double* opp;       // [S,max_opp,3] or null
    const int32_t* n_opp;    // [S] or null (-> max_opp)
    int max_opp;
    const double* lookaheads;  // [nL] device
    int nL;                    // 0 in explicit-goal mode
    int row0, row_step, n_rows;  // the lookahead rows this launch needs: row0 + k * row_step, k < n_rows
                                 // (a shard of a dense query samples only the rows it evaluates)
    QueryCtx* ctx;             // [S]
    Centre* centres;           // [S,nL]
    unsigned long long* best;  // [S]
    int* work_next;            // dense single query: the eval kernel's work counter, reset here (or null)
};

struct EvalArgs {
    TrackView tr;
    GridView grid;
    LutView lut;
    EvalParams ep;
    const QueryCtx* ctx;
    const Centre* centres;
    const float* widths;     // [nW] device
    int nL, nW;
    const float4* goals;     // explicit goals [S,C] (gx, gy, gth, p3) or null
    const float* prev_theta; // previous path of scenario s at prev_theta + s * prev_stride, or null
    int prev_stride;         // 0: one [M] path for every scenario (single query), M: [S,M]
    const uint8_t* prev_valid; // [S]: scenario s has a previous path iff != 0 (null: every one has)
    const float* weights;    // [S,5] cost weights of each scenario (the PW instances only)
    int C;                   // candidates per scenario
    int c_begin, c_end;      // evaluated range (of shard-local indices when row_step > 1)
    int row0, row_step;      // row-interleaved shard: local index v -> lookahead row
                             // row0 + (v / nW) * row_step, same width column (row_step 1: c = v)
    int ctas_per_scn;        // CTAs per scenario
    int chunk;               // candidates per CTA
    int item;                // candidates a warp takes at a time: 4 (their Newton solves share the
                             // warp, cubic generator, >= 4 candidates per warp) or 1
    float inv_nW;            // 1 / nW (row = floor((c + 0.5) / nW) without an integer division)
    int nseg_pad;            // shared-memory window capacity (multiple of 32)
    // outputs (nullable)
    float* costs;            // [S,C]
    float* terms;            // [S,C,5]
    uint8_t* flags;          // [S,C]
    float* goals_out;        // [S,C,3]
    float4* params;          // [S,C]
    float4* states;          // [S,C,M]
    float2* headings;        // [S,C,M] (cos, sin) used by the footprint (teacher-forced tests)
    unsigned long long* best;  // [S]
    unsigned long long* stats; // [2] deviation-pass work counters (segment steps, candidates) or null
    int* work_next;          // dense single query on a persistent grid: every warp pulls its next
                             // candidate from this device-wide counter (null: the CTA's own chunk)
    int v_last;              // with work_next: the walk is reversed, v -> v_last - v (far lookahead
                             // rows, the expensive candidates, first; the cheap ones fill the tail)
    // moving opponents (the MO instances only)
    const double* opp_vel;   // [S,vel_stride,2] map-frame opponent velocities (vx, vy), m/s, finite
    int vel_stride;          // opponent slots per scenario in opp_vel
    double v_min;            // the ego is timed at max(pose speed, v_min) along its candidate
    float* mo_ctx;           // [1 + 2 F1L_MAX_OPP] k_t and the vehicle-frame (wx, wy) of scenario 0,
                             // written by its first CTA (debug, nullable)
};

// Peer-memory exchange of a candidate-sharded query (SURVEY 8e: the one exchange step of the
// path).  Every rank owns a block of u64 words in its HBM, mapped into the other ranks' address
// spaces with CUDA IPC (NVLink P2P):
//   [0] call sequence number (local)     [1] sticky timeout flag (local)
//   [2..5] arrival counters of the four round-robin slots
//   [8 + (slot * F1L_MAX_RANKS + r) * 6 ...] entry of rank r in that slot: the rank's packed
//        (cost, index) key and the goal centre (Centre, 32 bytes) of its winner -- the winner's
//        lookahead row was sampled by its owner only, so the centre travels with the key.
#define F1L_MAX_RANKS 16
#define F1L_XCHG_ENTRY 6                                         // words per entry (key, Centre, pad)
#define F1L_XCHG_ENTRY0 8
#define F1L_XCHG_WORDS (F1L_XCHG_ENTRY0 + 4 * F1L_MAX_RANKS * F1L_XCHG_ENTRY)
#ifndef F1L_XCHG_TIMEOUT_CYCLES
#define F1L_XCHG_TIMEOUT_CYCLES 4000000000ll   // ~2 s at 1.965 GHz: a dead peer must not hang the GPU
#endif
struct XchgView {
    int world, rank;                                // world <= 1: no exchange
    unsigned long long* peer[F1L_MAX_RANKS];        // peer[rank] is the local block
};

// Lanes r < world each store this rank's (key, centre) entry into rank r's block over NVLink,
// fence, then bump rank r's arrival counter; lane 0 waits until all `world` arrivals are visible in
// the local block, then the lanes read the `world` keys and the warp takes their minimum -- every
// rank ends with the same key, the first minimum of the concatenated cost vector (np.argmin), and
// the centre its owner sent along.  Slots are used round-robin by call number and a call resets
// the counter of the slot two calls ahead: a peer can only be one call ahead of the slowest rank
// (it waits for everybody's arrival), so a slot is never reset while somebody may still write or
// read it.  Returns the global key and overwrites `ce` with the winner's centre; *timed_out is
// set when a peer did not arrive within F1L_XCHG_TIMEOUT_CYCLES.
__device__ __forceinline__ unsigned long long xchg_global_min(const XchgView& xc, unsigned long long key,
                                                              Centre& ce, int lane, int* timed_out) {
    unsigned long long* mine = xc.peer[xc.rank];
    const unsigned seq = (unsigned)(*(volatile unsigned long long*)(mine + 0));
    const int slot = (int)(seq & 3u);
    if (lane < xc.world) {
        volatile unsigned long long* dst =
            xc.peer[lane] + F1L_XCHG_ENTRY0 + (slot * F1L_MAX_RANKS + xc.rank) * F1L_XCHG_ENTRY;
        const unsigned long long* cw = reinterpret_cast<const unsigned long long*>(&ce);
        dst[0] = key;
        dst[1] = cw[0]; dst[2] = cw[1]; dst[3] = cw[2]; dst[4] = cw[3];
        __threadfence_system();
        atomicAdd_system(xc.peer[lane] + 2 + slot, 1ull);
    }
    __syncwarp();
    int bad = 0;
    if (lane == 0) {
        const long long t0 = clock64();
        volatile unsigned long long* cnt = mine + 2 + slot;
        while (*cnt < (unsigned long long)xc.world) {
            if (clock64() - t0 > F1L_XCHG_TIMEOUT_CYCLES) { bad = 1; break; }
        }
        __threadfence_system();
    }
    __syncwarp();
    // the world keys, one per lane; 64-bit minimum over the warp, the lowest rank on ties (keys of
    // different ranks differ in their index part unless both are ~0)
    const volatile unsigned long long* ent = mine + F1L_XCHG_ENTRY0 + (size_t)slot * F1L_MAX_RANKS * F1L_XCHG_ENTRY;
    unsigned long long k = lane < xc.world ? ent[lane * F1L_XCHG_ENTRY] : ~0ull;
    unsigned long long g = k;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(F1L_FULL, g, o);
        g = other < g ? other : g;
    }
    const unsigned who = __ballot_sync(F1L_FULL, lane < xc.world && k == g);
    const int wr = who ? __ffs(who) - 1 : xc.rank;
    if (wr != xc.rank) {   // warp-uniform
        unsigned long long* cw = reinterpret_cast<unsigned long long*>(&ce);
        const volatile unsigned long long* src = ent + wr * F1L_XCHG_ENTRY;
        cw[0] = src[1]; cw[1] = src[2]; cw[2] = src[3]; cw[3] = src[4];
    }
    __syncwarp();
    if (lane == 0) {
        const int nxt = (slot + 2) & 3;
        mine[2 + nxt] = 0ull;
        mine[0] = (unsigned long long)(seq + 1u);
        if (bad) mine[1] = 1ull;
        bad |= (int)(*(volatile unsigned long long*)(mine + 1));
    }
    *timed_out = __shfl_sync(F1L_FULL, bad, 0);
    return g;
}

struct SelectArgs {
    XchgView xc;            // sharded single query: global argmin over the ranks' shards
    int32_t* xchg_status;   // [1] != 0: a peer did not arrive (nullable)
    TrackView tr;
    LutView lut;
    EvalParams ep;
    const QueryCtx* ctx;
    const Centre* centres;
    const float* widths;
    int nL, nW;
    float inv_nW;
    int row0, row_step, n_rows; // the lookahead rows this rank's sampler filled (see SampleArgs)
    const float4* goals;
    int C, c_begin;
    const unsigned long long* best;
    // outputs (nullable)
    int32_t* best_idx;      // [S]
    float* best_cost;       // [S]
    int32_t* status;        // [S,2] no_feasible, tracker_found
    double* steer_speed;    // [S,2]
    float4* best_traj;      // [S,M]
    double* best_traj_map;  // [S,M,4] map frame (X, Y, v, Theta): SURVEY B.8, closed-loop tracking
    float* prev_theta_out;  // [S,M] theta column of best_traj (update_prev)
    uint8_t* prev_valid_out; // [S] set to 1 (update_prev with per-scenario flags)
};

// Candidate index of shard-local index v.  A row-interleaved shard (rank r of W takes lookahead
// rows r, r + W, ...: near and far goals cost differently, contiguous blocks would leave the ranks
// unbalanced) walks local indices v = 0 .. n_rows * nW - 1; the candidate keeps its global index
// c = row * nW + column, so costs / flags land where the unsharded query puts them and the
// argmin key orders like np.argmin on the whole cost vector.
__device__ __forceinline__ int shard_candidate(int v, int nW, float inv_nW, int row0, int row_step) {
    if (row_step == 1) return v;   // uniform
    const int rv = __float2int_rd(((float)v + 0.5f) * inv_nW);
    return v + (row0 + rv * (row_step - 1)) * nW;
}

// goal of candidate c of scenario s (SURVEY B.1): centre + width * normal, or the explicit goal
__device__ __forceinline__ void candidate_goal(const Centre* __restrict__ centres,
                                               const float* __restrict__ widths,
                                               const float4* __restrict__ goals, int nL, int nW,
                                               float inv_nW, int C, int s, int c,
                                               bool use_goal_kappa, float& gx,
                                               float& gy, float& gth, float& p3, bool& have_centre,
                                               float& v_ref) {
    if (goals) {
        const float4 g = __ldg(goals + (size_t)s * C + c);
        gx = g.x; gy = g.y; gth = g.z; p3 = g.w;
        have_centre = true;
        v_ref = -1.0f;
    } else {
        // (c + 0.5) / nW is at least 0.5 / nW away from an integer: exact in FP32 for c < 2^22
        const int row = __float2int_rd(((float)c + 0.5f) * inv_nW), k = c - row * nW;
        const Centre* ce = centres + (size_t)s * nL + row;
        const float4 a = __ldg(reinterpret_cast<const float4*>(ce));
        const float4 b = __ldg(reinterpret_cast<const float4*>(ce) + 1);
        const float wk = __ldg(widths + k);
        gx = fmaf(wk, b.x, a.x);
        gy = fmaf(wk, b.y, a.y);
        gth = a.z;
        p3 = use_goal_kappa ? a.w : 0.0f;
        have_centre = b.w != 0.0f;
        v_ref = b.z;
    }
}

// ---------------------------------------------------------------------------------------------
// K2: sampler
// ---------------------------------------------------------------------------------------------
#define SAMPLE_THREADS 256        // batches of a few queries
#define SAMPLE_THREADS_MAX 1024   // a single query gets one warp per ~2 lookahead rows

// a wrapped into [-pi, pi): (a + pi) mod 2 pi - pi without the iterative fmod
__device__ __forceinline__ double wrap_to_pi64(double a) {
    const double two_pi = 6.283185307179586476925286766559, pi = 3.14159265358979323846;
    const double b = a + pi;
    double r = b - two_pi * floor(b * (1.0 / two_pi));
    if (r < 0.0) r += two_pi;
    if (r >= two_pi) r -= two_pi;
    return r - pi;
}

// goal centre of one lookahead row from its intersect_point result (lattice_planner.py:251: the
// segment-start waypoint's x, y, psi), in the vehicle frame
__device__ __forceinline__ Centre centre_from_hit(const TrackView& tr, const Intersect64& ip, double px,
                                                  double py, double pth, double cth, double sth) {
    Centre ce;
    const int r = ip.found ? pymod(ip.i, tr.n) : 0;
    const double2 c = tr.xy[r];
    const double psi = tr.psi[r];
    const double dx = c.x - px, dy = c.y - py;
    const double prel = wrap_to_pi64(psi - pth);
    ce.cx = ip.found ? (float)(cth * dx + sth * dy) : 0.0f;
    ce.cy = ip.found ? (float)(-sth * dx + cth * dy) : 0.0f;
    ce.psi_rel = ip.found ? (float)prel : 0.0f;
    ce.kappa_g = (float)tr.kappa[r];
    double sp_, cp_;
    sincos(prel, &sp_, &cp_);
    ce.nx = ip.found ? (float)(-sp_) : 0.0f;
    ce.ny = ip.found ? (float)cp_ : 0.0f;
    ce.v = (float)tr.v[r];
    ce.ok = ip.found ? (float)(r + 1) : 0.0f;   // centre waypoint index + 1 (exact: < 2^24)
    return ce;
}

// everything after the nearest-point search, shared by the two sampler kernels.  `lt` / `nt`:
// this thread's index / the number of threads working on scenario s.
// `d_ego`: the float64 distance of the pose to its nearest raceline point (nearest_point's third
// result).
__device__ __forceinline__ void sample_body(const SampleArgs& a, int s, int lt, int nt, int i_ego,
                                            double t_ego, double d_ego) {
    const double px = a.poses[4 * (size_t)s], py = a.poses[4 * (size_t)s + 1];
    const double pth = a.poses[4 * (size_t)s + 2], pv = a.poses[4 * (size_t)s + 3];
    const int nseg = a.tr.n - 1;
    double cth, sth;
    sincos(pth, &sth, &cth);

    // one intersect_point per lookahead row (lattice_planner.py:249-251); an 8-lane group per row,
    // four rows per warp at a time
    XYTrack acc{a.tr.xy};
    const int lane = lt & 31;
    const int n_rows = a.nL > 0 ? a.n_rows : 0;
    for (int j0 = (lt >> 5) * 4; j0 < n_rows; j0 += (nt >> 5) * 4) {
        const int jj = j0 + (lane >> 3);
        const bool active = jj < n_rows;
        const int j = a.row0 + (active ? jj : j0) * a.row_step;   // lookahead row
        const double L = a.lookaheads[j];
        const TrackPrefilter pf = track_prefilter(a.tr, px, py, L);
        // A circle that stays clear of the raceline -- the pose is farther from its nearest
        // raceline point than the lookahead (2 mm of slack over the FP32 pre-scan behind d_ego) --
        // cannot cross any open segment: no scan, only the closing segment's test.  (18 % of the
        // benchmark's scenarios at L = 0.4 m; the scan would walk the whole track to find nothing.)
        const bool clear = active && d_ego > L + 2e-3;
        bool pending;
        Intersect64 ip = intersect_point_group<8>(acc, a.tr.n, px, py, L, (double)i_ego + t_ego,
                                                  true, lane, pf, active && !clear, 4, pending);
        if (__any_sync(F1L_FULL, clear)) {
            const Intersect64 co = intersect_closing_only(acc, a.tr.n, px, py, L, true);
            if (clear) ip = co;
        }
        // rows whose hit is not within the first 32 segments: the full 32-lane scan from there on,
        // one row after the other
        for (unsigned open = __ballot_sync(F1L_FULL, pending) & 0x01010101u; open; open &= open - 1) {
            const int src = __ffs(open) - 1;
            const double Ls = __shfl_sync(F1L_FULL, L, src);
            const TrackPrefilter pfs = track_prefilter(a.tr, px, py, Ls);
            const Intersect64 full =
                intersect_point_warp(acc, a.tr.n, px, py, Ls, (double)i_ego + t_ego, true, lane, pfs, 32);
            if ((lane & ~7) == src) ip = full;
        }
        if (active && (lane & 7) == 0)
            a.centres[(size_t)s * a.nL + j] = centre_from_hit(a.tr, ip, px, py, pth, cth, sth);
    }

    QueryCtx* q = a.ctx + s;
    const int n_opp = a.opp ? (a.n_opp ? min(a.n_opp[s], a.max_opp) : a.max_opp) : 0;
    // only the n_opp entries in use are written (and read back by eval_kernel): the other slots of
    // the 16-entry table would be 2 x 256 bytes of HBM traffic per scenario for nothing
    for (int k = lt; k < n_opp; k += nt) {
        const double* op = a.opp + 3 * ((size_t)s * a.max_opp + k);
        const double dx = op[0] - px, dy = op[1] - py, ph = op[2] - pth;
        double so_, co_;
        sincos(ph, &so_, &co_);
        q->opp[k] = make_float4((float)(cth * dx + sth * dy), (float)(-sth * dx + cth * dy), (float)co_,
                                (float)so_);
    }
    if (lt == nt - 1) {
        q->px = px; q->py = py; q->th = pth; q->vel = pv;
        q->cth = (float)cth; q->sth = (float)sth;
        q->i_ego = i_ego;
        q->t_ego = t_ego;
        q->pad1 = 0.0;
        int ns = a.ep.window;
        if (ns <= 0 || ns > nseg) ns = nseg;
        q->nseg = ns;
        q->seg0 = pymod(i_ego - ns / 4, nseg);
        q->n_opp = n_opp;
        q->has_grid = a.grid.occ != nullptr;
        q->pad0 = 0;
        if (a.grid.occ) {
            const double bx = (px - a.grid.ox) * a.grid.inv_res, by = (py - a.grid.oy) * a.grid.inv_res;
            const double fx = floor(bx), fy = floor(by);
            q->gix = (int)fx; q->giy = (int)fy;
            q->gfx = (float)(bx - fx); q->gfy = (float)(by - fy);
            q->gA00 = (float)(cth * a.grid.inv_res); q->gA01 = (float)(-sth * a.grid.inv_res);
            q->gA10 = (float)(sth * a.grid.inv_res); q->gA11 = (float)(cth * a.grid.inv_res);
        } else {
            q->gix = 0; q->giy = 0; q->gfx = 0.f; q->gfy = 0.f;
            q->gA00 = 0.f; q->gA01 = 0.f; q->gA10 = 0.f; q->gA11 = 0.f;
        }
        a.best[s] = ~0ull;
    }
}

// single / few queries: one CTA per scenario; nearest_point (utils.py:37-67) as a CTA-parallel
// FP32 scan of the block-local line form + float64 re-evaluation of the winner's neighbours.
__global__ void __launch_bounds__(SAMPLE_THREADS_MAX) sample_kernel(SampleArgs a) {
    __shared__ float s_d[SAMPLE_THREADS_MAX / 32];
    __shared__ int s_i[SAMPLE_THREADS_MAX / 32];
    __shared__ double s_t, s_dist;
    __shared__ int s_best;
    const int s = blockIdx.x;
    const int nthreads = blockDim.x;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const double px = a.poses[4 * (size_t)s], py = a.poses[4 * (size_t)s + 1];
    const int nseg = a.tr.n - 1;
    if (a.work_next && s == 0 && tid == 0) *a.work_next = 0;

    float bd = CUDART_INF_F;
    int bi = 0x7fffffff;
    for (int k = tid; k < nseg; k += nthreads) {
        const double2 o = a.tr.blk_origin[k >> 5];
        const float prx = (float)(px - o.x) * TRACK_SCALE, pry = (float)(py - o.y) * TRACK_SCALE;
        const float d2 = track_seg_d2(prx, pry, __ldg(a.tr.segA + k), __ldg(a.tr.segB + k));
        if (d2 < bd) { bd = d2; bi = k; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(F1L_FULL, bd, o);
        const int oi = __shfl_xor_sync(F1L_FULL, bi, o);
        if (od < bd || (od == bd && oi < bi)) { bd = od; bi = oi; }
    }
    if (lane == 0) { s_d[wid] = bd; s_i[wid] = bi; }
    __syncthreads();
    if (wid == 0) {   // warp 0: the warps' minima (one per lane), then the float64 neighbours on five lanes
        const int nw = nthreads >> 5;
        bd = lane < nw ? s_d[lane] : CUDART_INF_F;
        bi = lane < nw ? s_i[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float od = __shfl_xor_sync(F1L_FULL, bd, o);
            const int oi = __shfl_xor_sync(F1L_FULL, bi, o);
            if (od < bd || (od == bd && oi < bi)) { bd = od; bi = oi; }
        }
        if (bi == 0x7fffffff) bi = 0;
        const Nearest64 nr = refine_nearest64_warp(a.tr.xy, nseg, px, py, bi, lane);
        if (lane == 0) {
            s_best = nr.i;
            s_t = nr.t;
            s_dist = nr.dist;
        }
    }
    __syncthreads();
    sample_body(a, s, tid, nthreads, s_best, s_t, s_dist);
}

// batches: the nearest-point search of all scenarios is done by pp_scan_kernel + pp_finish_kernel (K1, lane per pose,
// track in shared memory); here one warp per scenario does the rest.
#define SAMPLE_WARPS 4
__global__ void __launch_bounds__(SAMPLE_WARPS * 32)
sample_warp_kernel(SampleArgs a, const int32_t* __restrict__ near_i,
                   const double* __restrict__ near4, int n_scenarios) {
    const int s = blockIdx.x * SAMPLE_WARPS + (threadIdx.x >> 5);
    if (s >= n_scenarios) return;
    sample_body(a, s, threadIdx.x & 31, 32, near_i[s], near4[4 * (size_t)s + 3], near4[4 * (size_t)s + 2]);
}

// ---------------------------------------------------------------------------------------------
// K3 + K4: fused generate / cost / collision, one warp per candidate
// ---------------------------------------------------------------------------------------------
#define EVAL_MAX_WARPS 8

// collision predicate pieces use explicitly rounded FP32 ops (no implicit FMA contraction; the
// sample -> grid-cell transform is written as explicit fused multiply-adds, fmaf in the mirror) so
// that the float32 mirror in the oracle reproduces the flags bit for bit on identical inputs.
__device__ __forceinline__ float ffm(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ float fm(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fs(float a, float b) { return __fsub_rn(a, b); }
// the same in float64: the rollout kernel (f1l_rollout.cuh) runs the predicates below in the map frame
__device__ __forceinline__ double fm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double fa(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double fs(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float vabs(float a) { return fabsf(a); }
__device__ __forceinline__ double vabs(double a) { return fabs(a); }
__device__ __forceinline__ int floor_int(float a) { return __float2int_rd(a); }
__device__ __forceinline__ int floor_int(double a) { return __double2int_rd(a); }

// SAT of two equal rectangles; ego axes (c, s), opponent axes (oc, os), T = opp - ego.
// collide iff every axis overlaps strictly (touching = no collision).
template <class T>
__device__ __forceinline__ bool sat_collide(T tx, T ty, T c, T s, T oc, T os, T hl, T hw) {
    const T cc = vabs(fa(fm(c, oc), fm(s, os)));
    const T ss = vabs(fs(fm(s, oc), fm(c, os)));
    const T rl = fa(hl, fa(fm(hl, cc), fm(hw, ss)));
    const T rw = fa(hw, fa(fm(hl, ss), fm(hw, cc)));
    const T e0 = vabs(fa(fm(tx, c), fm(ty, s)));
    const T e1 = vabs(fs(fm(ty, c), fm(tx, s)));
    const T e2 = vabs(fa(fm(tx, oc), fm(ty, os)));
    const T e3 = vabs(fs(fm(ty, oc), fm(tx, os)));
    return e0 < rl && e1 < rw && e2 < rl && e3 < rw;
}

// occupancy probe at cell (ix0 + floor(cx), iy0 + floor(cy)); out of bounds counts as occupied
template <class T>
__device__ __forceinline__ bool grid_hit(const uint8_t* __restrict__ occ, int gw, int gh, int ix0,
                                         int iy0, T cx, T cy) {
    const int col = ix0 + floor_int(cx), row = iy0 + floor_int(cy);
    if ((unsigned)col >= (unsigned)gw || (unsigned)row >= (unsigned)gh) return true;
    return __ldg(occ + (size_t)row * gw + col) != 0;
}

__device__ __forceinline__ float fast_sqrt(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Raceline deviation: distance of a sample to one window segment in line form.  The segment's
// table entry is T0 = (ux, uy, -uy, 1/len), T1 = (-(a.u + h), -a.n, -h, 0) with h = len / 2, so
// that q = p.u - (a.u + h) is measured from the segment's midpoint and n = p.n - a.n; the
// distance beyond the segment's ends is
//   e = sat(|q| - h)
// and d^2 = e^2 + n^2 (nearest_point, utils.py:53-65, without the division and the square root).
// (Nothing reads T0.w; the entry keeps it.)  e is one FADD.SAT with an |.| operand modifier: no ALU instruction and the fewest
// register-operand reads of the formulations measured (DESIGN §8, profiles/r2_microbench.md).
// The loop is bound by register-file operand bandwidth (about two 32-bit operands per lane per
// clock, measured: tools/microbench/rf_bench.cu), not by the FMA pipe, so operand reads count.
// Samples and table hold all lengths in units of EVAL_DEV_UNIT metres so that the saturation
// (clamp to [0, 1]) only ever acts at 0.
constexpr float EVAL_DEV_UNIT = 16384.0f;   // metres per table unit (a power of two: the scaling is exact)
constexpr float EVAL_DEV_SCALE = 1.0f / EVAL_DEV_UNIT;
#define EVAL_SEG_PAD 32   // readable slack behind the window tables (software-pipelined loads)

// e of a packed pair from its q
__device__ __forceinline__ f32x2 seg_axis_excess(f32x2 q2, const float4& T1) {
    float qa, qb;
    unpack2(q2, qa, qb);
    return pack2(__saturatef(fabsf(qa) + T1.z), __saturatef(fabsf(qb) + T1.z));
}

// squared distance of one sample (sx, sy) to one window segment (table units)
__device__ __forceinline__ float seg_dist2(float sx, float sy, const float4& T0, const float4& T1) {
    const float qq = fmaf(sx, T0.x, fmaf(sy, T0.y, T1.x));
    const float nn = fmaf(sy, T0.x, fmaf(sx, T0.z, T1.y));
    const float e = __saturatef(fabsf(qq) + T1.z);
    return fmaf(e, e, nn * nn);
}

// Squared distances of the sample pairs [J0, J0 + EVAL_DEV_GROUP) of a lane to one segment, on
// packed FP32x2 instructions whose segment constants enter as scalar-broadcast operands, in
// operation-major order: consecutive instructions share their segment constants, which then come
// from the operand reuse cache instead of the register file.  (Pairs per group, re-measured with
// the batch shape at 125 registers: 2 gives 10.76 ms against 10.83 on the full scan but 6.50
// against 6.35 with prune_window = 1; 6: 10.88.)
constexpr int EVAL_DEV_GROUP = 3;
template <int SP, int J0>
__device__ __forceinline__ void seg_group(const f32x2 (&sx2)[SP], const f32x2 (&sy2)[SP],
                                          const float4& T0, const float4& T1,
                                          f32x2 (&d)[EVAL_DEV_GROUP]) {
    const f32x2 ux = pack2(T0.x, T0.x), uy = pack2(T0.y, T0.y);
    const f32x2 nuy = pack2(T0.z, T0.z), nc = pack2(T1.x, T1.x), ne = pack2(T1.y, T1.y);
    f32x2 q[EVAL_DEV_GROUP], n[EVAL_DEV_GROUP], e[EVAL_DEV_GROUP];
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) q[j] = ffma2(sy2[J0 + j], uy, nc);
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) n[j] = ffma2(sx2[J0 + j], nuy, ne);
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) q[j] = ffma2(sx2[J0 + j], ux, q[j]);
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) n[j] = ffma2(sy2[J0 + j], ux, n[j]);
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) e[j] = seg_axis_excess(q[j], T1);
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) n[j] = fmul2(n[j], n[j]);
#pragma unroll
    for (int j = 0; j < EVAL_DEV_GROUP; ++j) if (J0 + j < SP) d[j] = ffma2(e[j], e[j], n[j]);
}

// running minima of all SP sample pairs of a lane over two segments A and B: the minimum takes
// both distances in one three-input FMNMX3
template <int SP, int J0 = 0>
__device__ __forceinline__ void seg_min2(const f32x2 (&sx2)[SP], const f32x2 (&sy2)[SP],
                                         const float4& A0, const float4& A1, const float4& B0,
                                         const float4& B1, float (&bdx)[SP], float (&bdy)[SP]) {
    if constexpr (J0 < SP) {
        f32x2 dA[EVAL_DEV_GROUP], dB[EVAL_DEV_GROUP];
        seg_group<SP, J0>(sx2, sy2, A0, A1, dA);
        seg_group<SP, J0>(sx2, sy2, B0, B1, dB);
#pragma unroll
        for (int j = 0; j < EVAL_DEV_GROUP; ++j)
            if (J0 + j < SP) {
                float da, db, ea, eb;
                unpack2(dA[j], da, db);
                unpack2(dB[j], ea, eb);
                bdx[J0 + j] = fmin3(bdx[J0 + j], da, ea);
                bdy[J0 + j] = fmin3(bdy[J0 + j], db, eb);
            }
        seg_min2<SP, J0 + EVAL_DEV_GROUP>(sx2, sy2, A0, A1, B0, B1, bdx, bdy);
    }
}

// Deviation-pass epilogue: v[r] (r < N) is this lane's running minimum of squared distance for
// row r of its sample group, of which the first `cnt` exist; the group's LANES lanes (consecutive,
// LANES a power of two) hold minima over different segments.  Halving butterfly: the lane whose
// bit is clear keeps the first half of the rows, its partner the second; after log2(LANES) steps
// every row is reduced on exactly one lane of the group.  Returns the sum of sqrt over this
// lane's existing rows, so that a plain warp sum gives the total over all samples.
template <int N, int LANES>
__device__ __forceinline__ float halve_min_sqrt_sum(float (&v)[N], int lane_in_group, int cnt) {
    if constexpr (LANES == 1) {
        float s = 0.0f;
#pragma unroll
        for (int j = 0; j < N; ++j) s += (j < cnt) ? fast_sqrt(v[j]) : 0.0f;
        return s;
    } else {
        constexpr int H = (N + 1) / 2;
        const bool hi = (lane_in_group & (LANES / 2)) != 0;
        float out[H];
#pragma unroll
        for (int j = 0; j < H; ++j) {
            const float lo_v = v[j];
            const float hi_v = (j + H < N) ? v[j + H] : CUDART_INF_F;
            const float keep = hi ? hi_v : lo_v;
            const float send = hi ? lo_v : hi_v;
            out[j] = fminf(keep, __shfl_xor_sync(F1L_FULL, send, LANES / 2));
        }
        // rows exist from the front: the first half holds min(cnt, H) of them, the second the rest
        return halve_min_sqrt_sum<H, LANES / 2>(out, lane_in_group, hi ? max(cnt - H, 0) : min(cnt, H));
    }
}

// Shared-memory layout of eval_kernel (bytes; the host sizes a launch as C_TAB plus the window
// table's (nseg_pad + EVAL_SEG_PAD) x 32 bytes).  Per warp one contiguous block -- list of the footprints that need their nine grid probes (centre and half-axes
// in grid-cell coordinates, two float4 per entry) | solutions of the four candidates of an item
// ((gx, gy, gth, p3), (p1, p2, sf, have | passes)) | sample slab x | sample slab y, in the pair
// layout of the deviation pass: element (j, sg, half) holds sample (2j + half) * SG + sg, so that
// one 64-bit load yields a packed pair of samples -- then the CTA-wide part: opponents | grid
// constants | previous path | window table (run-time length, last).  Everything sits at a
// compile-time offset from two addresses, the CTA's base and the warp's block.
template <int S, int SG, int NW, bool MO = false>
struct EvalSmem {
    static constexpr int PCAP = S * SG;
    static constexpr int SROWS = (S + 1) / 2;
    static constexpr int SLAB = SROWS * SG * 2;                    // floats per coordinate
    static constexpr uint32_t W_PLIST = 0;                         // [PCAP][2] float4
    static constexpr uint32_t W_ITEM = W_PLIST + PCAP * 32;        // [4][2] float4
    static constexpr uint32_t W_SLABX = W_ITEM + 128;              // [SLAB] float
    static constexpr uint32_t W_SLABY = W_SLABX + SLAB * 4;
    static constexpr uint32_t W_BYTES = W_SLABY + SLAB * 4;
    static constexpr uint32_t C_OPP = NW * W_BYTES;                // [F1L_MAX_OPP] float4
    static constexpr uint32_t C_GRID = C_OPP + F1L_MAX_OPP * 16;   // 4 float4: A, (fx, fy, ix0, iy0),
                                                                   // (n_opp, has_grid, use_prev, w4), (w0, w1, w2, w3)
                                                                   // (the weights with PW only)
    static constexpr uint32_t C_PREV = C_GRID + 64;                // [F1L_MAX_M] float
    static constexpr uint32_t C_VEL = C_PREV + F1L_MAX_M * 4;      // MO: [F1L_MAX_OPP] (wx, wy), k_t
    static constexpr uint32_t C_TAB = C_VEL + (MO ? F1L_MAX_OPP * 8 + 16 : 0);   // [ntab][2] float4
    static_assert(W_BYTES % 16 == 0, "per-warp block keeps 16-byte alignment");
};

// One CTA per (scenario, candidate chunk).  The CTA builds the scenario's raceline window once,
// then its NW warps pull candidates of the chunk from a shared counter until it is exhausted
// (warps that finish an early-exit candidate immediately take the next one).
// PW: the call has per-scenario cost weights (a.weights), which the candidate loop reads from the
// CTA's shared memory.  Without them the instance takes the config's weights from the kernel
// parameters, whose constant-bank operands cost no register: its schedule is the one it had before
// per-scenario weights existed (shared-memory operands there made the batch instance 1.2 % slower).
// MO (PW instances only): the opponents move at constant velocity.  Opponent k's centre at time t
// is o_k + w_k t (vehicle frame, heading kept); the ego reaches sample i of a candidate of length
// s_f at t_i = i * s_f * k_t, k_t = 1 / ((M - 1) v_e), v_e = max(pose speed, v_min).  The prologue
// stages k_t and the w_k next to the opponents; the prune, the broad phase and the narrow phase
// test the predicted centres.  With every velocity zero the flags are those of the PW instance,
// and a call without weights gives the config's weights as every scenario's row.
template <int IPL, int S, int SG, int NW, int MINB, bool PW, bool MO = false>
__global__ void __launch_bounds__(NW * 32, MINB) eval_kernel(EvalArgs a) {
    static_assert(!MO || PW, "the moving-opponent instances are twins of the PW instances");
    constexpr int GG = 32 / SG;
    using L = EvalSmem<S, SG, NW, MO>;
    extern __shared__ __align__(16) unsigned char ev_smem[];
    __shared__ int s_next;
    __shared__ unsigned long long s_work;   // deviation pass: candidates << 40 | (candidate, segment) pairs
    const int M = a.ep.M;
    const int ntab = a.nseg_pad + EVAL_SEG_PAD;
    constexpr int PCAP = L::PCAP;
    constexpr int SLAB = L::SLAB;

    int s, cta;
    // persistent grid over one dense query (never with the 4-warp CTAs of the batch regime: the
    // compile-time false keeps that instance's candidate loop free of the extra state)
    const bool dyn = NW != 4 && a.work_next != nullptr;
    if (a.ctas_per_scn == 1) { s = blockIdx.x; cta = 0; }
    else if (dyn) { s = 0; cta = 0; }
    else { s = blockIdx.x / a.ctas_per_scn; cta = blockIdx.x - s * a.ctas_per_scn; }
    const int tid = threadIdx.x, wid = tid >> 5;
    // The three values every shared access and every guard below derives from.  They go through
    // opaque() so that the compiler keeps (or spills) them instead of re-deriving each one at
    // every use from S2R / SR_CgaCtaId -- see f1l_common.cuh.
    int lane = tid & 31;
    uint32_t cbase = smem_u32(ev_smem);            // the CTA's dynamic shared memory
    uint32_t wbase = cbase + wid * L::W_BYTES;     // this warp's block
    int nown = min(max(M - lane * IPL, 0), IPL);   // samples [lane * IPL, lane * IPL + nown) exist
    opaque(lane);
    opaque(cbase);
    opaque(wbase);
    opaque(nown);
    const QueryCtx* __restrict__ q = a.ctx + s;
    const int cb = a.c_begin + cta * a.chunk;
    const int ce = dyn ? a.c_end : min(cb + a.chunk, a.c_end);

    // ---- prologue: raceline window -> vehicle frame -> line form in shared memory.  Only the
    //      subtraction of the pose happens in float64 (|coordinates| reach 85 m, the window is
    //      ~25 m long); rotation, length and line coefficients are FP32 on ego-relative values.
    {
        const double px = q->px, py = q->py;
        const float cth = q->cth, sth = q->sth;
        const int seg0 = q->seg0, nseg = q->nseg, ns = a.tr.n - 1;
        for (int k = tid; k < ntab; k += NW * 32) {
            float4 T0 = make_float4(1.0f, 0.0f, -0.0f, 1.0f);      // padding: far away, finite
            float4 T1 = make_float4(-1e9f, -1e9f, -1.0f, 0.0f);    // (table units) d^2 = 1e18
            if (k < nseg) {
                int sg = seg0 + k;
                if (sg >= ns) sg -= ns;
                const double2 p0 = a.tr.xy[sg], p1 = a.tr.xy[sg + 1];
                const float ax = (float)(p0.x - px), ay = (float)(p0.y - py);
                const float dxm = (float)(p1.x - p0.x), dym = (float)(p1.y - p0.y);
                const float avx = fmaf(cth, ax, sth * ay), avy = fmaf(cth, ay, -sth * ax);
                const float dx = fmaf(cth, dxm, sth * dym), dy = fmaf(cth, dym, -sth * dxm);
                const float l2 = fmaf(dx, dx, dy * dy);
                // a zero-length segment (a repeated waypoint) is its point: any unit direction,
                // h = 0.  (rsqrtf(0) would make the entry NaN, which the minima ignore, and the
                // point would drop out of a window it ends.)
                const bool point = !(l2 > 0.0f);
                const float il = point ? 0.0f : rsqrtf(l2);
                const float ux = point ? 1.0f : dx * il, uy = point ? 0.0f : dy * il;
                T0 = make_float4(ux, uy, -uy, il);
                const float hh = 0.5f * (l2 * il);
                T1 = make_float4(-(fmaf(avx, ux, avy * uy) + hh) * EVAL_DEV_SCALE,
                                 -fmaf(avy, ux, -avx * uy) * EVAL_DEV_SCALE, -hh * EVAL_DEV_SCALE, 0.0f);
            }
            sts128(cbase + L::C_TAB + k * 32, T0);
            sts128(cbase + L::C_TAB + k * 32 + 16, T1);
        }
        // the scenario's previous path (every CTA of a scenario loads its own copy)
        const bool use_prev = a.prev_theta && (!a.prev_valid || a.prev_valid[s]);
        if (use_prev) {
            const float* pt = a.prev_theta + (size_t)s * a.prev_stride;
#pragma unroll 1
            for (int i = tid; i < M; i += NW * 32) sts32(cbase + L::C_PREV + i * 4, pt[i]);
        }
        if (tid < F1L_MAX_OPP)   // unused slots: an opponent far away
            sts128(cbase + L::C_OPP + tid * 16,
                   tid < q->n_opp ? q->opp[tid] : make_float4(1e9f, 1e9f, 1.0f, 0.0f));
        if constexpr (MO) {
            // velocities rotated into the vehicle frame with the pose's float64 cos / sin, as the
            // sampler rotates the positions (unused slots: at rest)
            const bool dbg = a.mo_ctx && blockIdx.x == 0;
            if (tid < F1L_MAX_OPP) {
                float wx = 0.0f, wy = 0.0f;
                if (tid < q->n_opp) {
                    const double* vel = a.opp_vel + 2 * ((size_t)s * a.vel_stride + tid);
                    double sth, cth;
                    sincos(q->th, &sth, &cth);
                    wx = (float)fa(fm(cth, vel[0]), fm(sth, vel[1]));
                    wy = (float)fs(fm(cth, vel[1]), fm(sth, vel[0]));
                }
                sts32(cbase + L::C_VEL + tid * 8, wx);
                sts32(cbase + L::C_VEL + tid * 8 + 4, wy);
                if (dbg) { a.mo_ctx[1 + 2 * tid] = wx; a.mo_ctx[2 + 2 * tid] = wy; }
            }
            if (tid == F1L_MAX_OPP % (NW * 32)) {
                const double ve = fmax(q->vel, a.v_min);
                const float k_t = (float)__ddiv_rn(1.0, fm((double)(M - 1), ve));
                sts32(cbase + L::C_VEL + F1L_MAX_OPP * 8, k_t);
                if (dbg) a.mo_ctx[0] = k_t;
            }
        }
        if (tid == 0) { s_next = cb + NW * a.item; s_work = 0ull; }
        // per-scenario collision constants (and with PW the cost weights) live in shared memory,
        // not in registers, so that the candidate loop does not carry them through the deviation pass
        if (tid == 32 % (NW * 32)) {
            float w4 = 0.0f;
            if constexpr (PW) {
                // (a moving-opponent call without weights: the config's as the scenario's row)
                if (MO && !a.weights) {
                    w4 = a.ep.w[4];
                    sts128(cbase + L::C_GRID + 48, make_float4(a.ep.w[0], a.ep.w[1], a.ep.w[2], a.ep.w[3]));
                } else {
                    const float* w = a.weights + (size_t)s * F1L_N_TERMS;
                    w4 = w[4];
                    sts128(cbase + L::C_GRID + 48, make_float4(w[0], w[1], w[2], w[3]));
                }
            }
            sts128(cbase + L::C_GRID, make_float4(q->gA00, q->gA01, q->gA10, q->gA11));
            sts128(cbase + L::C_GRID + 16, make_float4(q->gfx, q->gfy, __int_as_float(q->gix), __int_as_float(q->giy)));
            sts128(cbase + L::C_GRID + 32, make_float4(__int_as_float(q->n_opp), __int_as_float(q->has_grid),
                                                       __int_as_float((int)use_prev), w4));
        }
    }
    __syncthreads();

#pragma unroll 1
    for (int i = M + lane; i < S * SG; i += 32) {   // unused slots of the last rows: finite dummies
        const int r = i / SG, g = i - r * SG;
        const uint32_t at = (uint32_t)(((r >> 1) * SG + g) * 2 + (r & 1)) * 4;
        sts32(wbase + L::W_SLABX + at, 0.0f);
        sts32(wbase + L::W_SLABY + at, 0.0f);
    }
    // deviation pass: this lane's sample group / segment group, and how many of the group's S
    // sample rows exist (row r holds sample r * SG + sgi; rows are valid from the front)
    const int sgi = lane / GG, ggi = lane - sgi * GG;
    int nrows = min(max((M - sgi + SG - 1) / SG, 0), S);
    opaque(nrows);

    // A warp takes `item` consecutive candidates at a time.  With item = 4 their goals, LUT seeds
    // and Newton solves run together, one candidate per 8-lane group (spiral_newton_g8); the rest
    // of the pipeline then handles the four one after the other on the whole warp.
    const int item = a.item;
    int c_first = cb + wid * item;
    if (dyn) {
        if (lane == 0) c_first = cb + atomicAdd(a.work_next, item);
        c_first = __shfl_sync(F1L_FULL, c_first, 0);
    }
    for (int c0 = c_first; c0 < ce;) {
      if (item == 4) {   // warp-uniform
          const int cg = c0 + (lane >> 3);
          const bool active = cg < ce;
          float ggx, ggy, ggth, gp3, gv_ref;
          bool ghave;
          const int cgv = active ? cg : c0;
          candidate_goal(a.centres, a.widths, a.goals, a.nL, a.nW, a.inv_nW, a.C, s,
                         shard_candidate(dyn ? a.v_last - cgv : cgv, a.nW, a.inv_nW, a.row0, a.row_step),
                         a.ep.use_goal_kappa != 0, ggx, ggy, ggth, gp3, ghave, gv_ref);
          SpiralF gsp;
          const int g_pass = generate_cubic_g8(gsp, a.lut, a.ep, ggx, ggy, ggth, gp3, lane, active);
          // through shared memory, not registers: nothing of this lives across the deviation pass
          if ((lane & 7) == 0) {
              const uint32_t ia = wbase + L::W_ITEM + 32 * (lane >> 3);
              sts128(ia, make_float4(ggx, ggy, ggth, gp3));
              sts128(ia + 16, make_float4(gsp.p1, gsp.p2, gsp.sf, __int_as_float((ghave ? 256 : 0) | g_pass)));
          }
          __syncwarp();
      }
      const int c_last = min(c0 + item, ce);
      for (int v = c0; v < c_last; ++v) {
        const int c = shard_candidate(dyn ? a.v_last - v : v, a.nW, a.inv_nW, a.row0, a.row_step);
        // ---- goal, seed, Newton ----
        float gx, gy, gth, p3, v_ref;
        bool have_centre;
        SpiralF sp;
        int n_pass;
        if (item == 4) {   // the solution of candidate c, found by its 8-lane group
            const uint32_t ia = wbase + L::W_ITEM + 32 * (v - c0);
            const float4 G = lds128(ia), Q = lds128(ia + 16);
            gx = G.x; gy = G.y; gth = G.z; p3 = G.w;
            v_ref = 0.0f;
            const int hp = __float_as_int(Q.w);
            have_centre = (hp & 256) != 0;
            n_pass = hp & 255;
            sp.p0 = 0.0f;
            sp.p3 = p3;
            sp.p1 = Q.x; sp.p2 = Q.y; sp.sf = Q.z;
            spiral_set(sp);
        } else {
            candidate_goal(a.centres, a.widths, a.goals, a.nL, a.nW, a.inv_nW, a.C, s, c,
                           a.ep.use_goal_kappa != 0, gx, gy, gth, p3, have_centre, v_ref);
            n_pass = generate_spiral(sp, a.lut, a.ep, gx, gy, gth, p3, lane);
        }

        // ---- arc samples ----
        float x[IPL], y[IPL], th[IPL], kp[IPL], cs[IPL], sn[IPL];
        spiral_sample<IPL>(sp, M, lane, x, y, th, kp, cs, sn);

        const size_t cand = (size_t)s * a.C + c;
        if (a.states) {
#pragma unroll
            for (int j = 0; j < IPL; ++j)
                if (j < nown) a.states[cand * M + lane * IPL + j] = make_float4(x[j], y[j], th[j], kp[j]);
        }
        if (a.headings) {
#pragma unroll
            for (int j = 0; j < IPL; ++j)
                if (j < nown) a.headings[cand * M + lane * IPL + j] = make_float2(cs[j], sn[j]);
        }

        // ---- curvature terms, endpoint, validity ----
        float maxk = 0.0f, sumk = 0.0f, ex = 0.0f, ey = 0.0f, eth = 0.0f;
        __syncwarp();   // the previous candidate's deviation pass has finished reading the slab
        {
            // slab address of this lane's first sample; when the IPL samples of a lane cannot
            // straddle a slab row (IPL divides SG) the others follow at 8-byte steps
            const int i0 = lane * IPL;
            const int r0 = i0 / SG, g0 = i0 - r0 * SG;
            const uint32_t wa = wbase + L::W_SLABX + (uint32_t)(((r0 >> 1) * SG + g0) * 2 + (r0 & 1)) * 4;
            const int last_lane = (M - 1) / IPL, last_j = (M - 1) - last_lane * IPL;   // uniform
#pragma unroll
            for (int j = 0; j < IPL; ++j) {
                if (j < nown) {
                    const float ak = fabsf(kp[j]);
                    maxk = fmaxf(maxk, ak);
                    sumk += ak;
                    uint32_t at = wa + 8 * j;
                    if constexpr (SG % IPL != 0) {
                        const int i = i0 + j, r = i / SG, g = i - r * SG;
                        at = wbase + L::W_SLABX + (uint32_t)(((r >> 1) * SG + g) * 2 + (r & 1)) * 4;
                    }
                    sts32(at, x[j] * EVAL_DEV_SCALE);
                    sts32(at + SLAB * 4, y[j] * EVAL_DEV_SCALE);
                }
                if (j == last_j) { ex = x[j]; ey = y[j]; eth = th[j]; }   // (uniform predicate)
            }
            ex = __shfl_sync(F1L_FULL, ex, last_lane);
            ey = __shfl_sync(F1L_FULL, ey, last_lane);
            eth = __shfl_sync(F1L_FULL, eth, last_lane);
        }
        maxk = warp_max(maxk);
        sumk = warp_sum(sumk);
        const float gn = sqrtf(fmaf(gx, gx, fmaf(gy, gy, gth * gth)));
        const float tol = a.ep.tol * fmaxf(gn, 1.0f);
        bool valid = have_centre && isfinite(sp.p1) && isfinite(sp.p2) && isfinite(sp.sf) &&
                     sp.sf > 0.0f && fabsf(ex - gx) < tol && fabsf(ey - gy) < tol &&
                     fabsf(eth - gth) < tol;
        if (valid && a.ep.kappa_max > 0.0f && !(maxk <= a.ep.kappa_max)) valid = false;

        unsigned flags = valid ? F1L_FLAG_VALID : 0u;
        if (!have_centre) flags |= F1L_FLAG_NO_CENTRE;
        flags |= (unsigned)min(n_pass, 15) << F1L_FLAG_PASS_SHIFT;
        // everything the deviation pass does not need leaves the registers before it starts:
        // goal / parameter outputs now, the first four cost terms as one partial sum
        if (lane == 0) {
            if (a.goals_out) {
                float* g = a.goals_out + cand * 3;
                g[0] = gx; g[1] = gy; g[2] = gth;
            }
            if (a.params)   // cubic: (p1, p2, s_f, p3); clothoid: (kappa0, dkappa, L, kappa_end)
                a.params[cand] = a.ep.generator == 1
                                     ? make_float4(sp.p0, __fdividef(sp.b1, sp.sf), sp.sf, sp.p3)
                                     : make_float4(sp.p1, sp.p2, sp.sf, sp.p3);
        }
        float t_dev = 0.0f, partial = 0.0f;
        float cost = CUDART_INF_F;

        if (valid) {  // warp-uniform
            const float t_len = __fdividef(1.0f, sp.sf);       // lattice_planner.py:271
            const float t_maxk = maxk;                         // :277
            const float t_meank = sumk * a.ep.inv_M;           // :284
            float t_sim = 0.0f;
            if constexpr (PW) {
                // the first three weighted terms now, so that only their sum lives through the
                // collision tests (the operations and order of the one weighted sum below)
                const float4 GW = lds128(cbase + L::C_GRID + 48);
                partial = GW.x * t_len + GW.y * t_maxk + GW.z * t_meank;
                if (lane == 0 && a.terms) {
                    float* t = a.terms + cand * F1L_N_TERMS;
                    t[0] = t_len; t[1] = t_maxk; t[2] = t_meank;
                }
            }

            // ---- similarity (lattice_planner.py:287-296), collision (SURVEY B.6) ----
            float sim = 0.0f;
            bool hit_opp = false, hit_map = false;
            const uint8_t* occ = a.grid.occ;
            const int gw = a.grid.w, gh = a.grid.h;
            const float4 GA = lds128(cbase + L::C_GRID), GB = lds128(cbase + L::C_GRID + 16);
            const float4 GC = lds128(cbase + L::C_GRID + 32);
            const int n_opp = __float_as_int(GC.x);
            const bool has_grid = __float_as_int(GC.y) != 0;
            const bool use_prev = __float_as_int(GC.z) != 0;
            const float hl = a.ep.half_l, hw = a.ep.half_w;
            const float A00 = GA.x, A01 = GA.y, A10 = GA.z, A11 = GA.w;
            const float gfx = GB.x, gfy = GB.y;
            const int gix = __float_as_int(GB.z), giy = __float_as_int(GB.w);
            // clearance map: clear[cell] = Chebyshev distance (cells) to the nearest occupied /
            // out-of-bounds cell.  All nine probes fall within `probe_reach` cells of the
            // footprint-centre cell, so a larger clearance proves them free without touching
            // them.  The loads are issued first, the opponent tests cover their latency.
            // (collision_mode 1, three discs on the Euclidean distance transform, works the same
            // way: the squared distance at the footprint centre's cell, when at least near_free,
            // proves all three discs free.)
            int clr[IPL];
#pragma unroll
            for (int j = 0; j < IPL; ++j) {
                clr[j] = 0;
                if (has_grid && a.grid.near_map && j < nown) {
                    const float ccx = ffm(A00, x[j], ffm(A01, y[j], gfx));
                    const float ccy = ffm(A10, x[j], ffm(A11, y[j], gfy));
                    const int ccol = gix + __float2int_rd(ccx), crow = giy + __float2int_rd(ccy);
                    if ((unsigned)ccol < (unsigned)gw && (unsigned)crow < (unsigned)gh)
                        clr[j] = __ldg(a.grid.near_map + (size_t)crow * gw + ccol);
                }
            }
            // candidate-level opponent pruning: every point of a curve of length s_f from the
            // origin to (ex, ey) lies within s_f/2 of the chord's midpoint, so an opponent
            // farther than s_f/2 + 2 r_circ from it cannot pass the per-sample broad phase.
            // MO: the ego reaches sample i at t_i = fm(i, dt).  Over [0, T], T = t_{M-1}, an
            // opponent's centre stays within |w| T / 2 of o + w T / 2: the reach grows by that
            // much, with 0.1 % + 1 mm of slack over the FP32 rounding of the predicted centres.
            float dt = 0.0f;
            if constexpr (MO) dt = fm(sp.sf, lds32(cbase + L::C_VEL + F1L_MAX_OPP * 8));
            unsigned opp_mask;
            {
                const float4 o = lds128(cbase + L::C_OPP + (lane & (F1L_MAX_OPP - 1)) * 16);
                float mx = o.x - 0.5f * ex, my = o.y - 0.5f * ey;
                float reach = 0.5f * sp.sf + a.ep.reach_pad;
                if constexpr (MO) {
                    float wx, wy;
                    unpack2(lds64(cbase + L::C_VEL + (lane & (F1L_MAX_OPP - 1)) * 8), wx, wy);
                    const float hT = 0.5f * fm((float)(M - 1), dt);
                    mx = fmaf(wx, hT, mx);
                    my = fmaf(wy, hT, my);
                    reach = fmaf(hT, sqrtf(fmaf(wx, wx, wy * wy)), reach) * 1.001f + 1e-3f;
                }
                opp_mask = __ballot_sync(F1L_FULL, lane < n_opp && fmaf(mx, mx, my * my) <= reach * reach);
            }
            if (use_prev) {   // uniform
                const int lim = M - a.ep.n_shift - a.ep.n_cull;
#pragma unroll
                for (int j = 0; j < IPL; ++j) {
                    const int i = lane * IPL + j;
                    if (i < lim) {
                        const float d = th[j] - lds32(cbase + L::C_PREV + (i + a.ep.n_shift) * 4);
                        sim = fmaf(d, d, sim);
                    }
                }
            }
            // lane-level broad phase: a lane's samples are consecutive points of the curve, so they
            // lie within (IPL - 1) arc steps of its first one; an opponent farther than that plus
            // the broad-phase radius from the first sample cannot pass any per-sample test.  (1 %
            // and 1 mm of slack over the quadrature; only provably negative tests are skipped,
            // the flags stay as they were.)
            // MO: over the lane's times [t_a, t_b] the opponent stays within |w| (t_b - t_a) / 2 of
            // its centre at (t_a + t_b) / 2 (same slack as the prune).
            float lane_R2 = -1.0f, lane_R = 0.0f;
            if (opp_mask && nown > 0) {
                const float R = fmaf(1.01f * (float)(IPL - 1), __fdividef(sp.sf, (float)(M - 1)), a.ep.reach_pad);
                lane_R2 = R * R;
                lane_R = R;
            }
            for (unsigned m = opp_mask; m; m &= m - 1) {   // uniform; mostly empty
                const int k = __ffs(m) - 1;
                const float4 o = lds128(cbase + L::C_OPP + k * 16);
                float wx = 0.0f, wy = 0.0f;
                float ux = o.x - x[0], uy = o.y - y[0];
                float R2 = lane_R2;
                if constexpr (MO) {
                    unpack2(lds64(cbase + L::C_VEL + k * 8), wx, wy);
                    const float ta = fm((float)(lane * IPL), dt), tb = fm((float)(lane * IPL + IPL - 1), dt);
                    const float tm = 0.5f * (ta + tb), hs = 0.5f * (tb - ta);
                    ux = fmaf(wx, tm, ux);
                    uy = fmaf(wy, tm, uy);
                    const float Rm = fmaf(hs, sqrtf(fmaf(wx, wx, wy * wy)), lane_R) * 1.001f + 1e-3f;
                    R2 = lane_R2 < 0.0f ? -1.0f : Rm * Rm;
                }
                if (fmaf(ux, ux, uy * uy) <= R2) {
#pragma unroll
                    for (int j = 0; j < IPL; ++j) {
                        if (j < nown) {
                            float cx = o.x, cy = o.y;   // the opponent's centre when the ego is at sample i
                            if constexpr (MO) {
                                const float t = fm((float)(lane * IPL + j), dt);
                                cx = fa(o.x, fm(wx, t));
                                cy = fa(o.y, fm(wy, t));
                            }
                            const float tx = fs(cx, x[j]), ty = fs(cy, y[j]);
                            const float d2 = fa(fm(tx, tx), fm(ty, ty));
                            if (d2 <= a.ep.rc2 && sat_collide(tx, ty, cs[j], sn[j], o.z, o.w, hl, hw))
                                hit_opp = true;
                        }
                    }
                }
            }
            if (has_grid) {
                // Samples whose clearance does not prove the footprint free get their nine probes.
                // They are few and scattered over the lanes (walls are near the outer goals
                // only), so the warp shares them: each owner lane writes the footprint of its
                // needy samples into a per-warp list, then all 32 lanes take (footprint, probe)
                // pairs from it -- ~6x fewer instructions than every lane probing its own
                // samples while the others idle.
                unsigned nm[IPL];
                int total = 0;
#pragma unroll
                for (int j = 0; j < IPL; ++j) {
                    nm[j] = __ballot_sync(F1L_FULL, j < nown && clr[j] < a.grid.near_free);
                    total += __popc(nm[j]);
                }
                if (total) {   // warp-uniform
                    const uint32_t pl = wbase + L::W_PLIST;
                    int rank0 = 0;
                    const bool discs = a.ep.collision_mode == 1;     // uniform
                    const float al = discs ? a.grid.disc_off : hl;   // extent along the body axis
#pragma unroll
                    for (int j = 0; j < IPL; ++j) {
                        if ((nm[j] >> lane) & 1u) {
                            const int r = rank0 + __popc(nm[j] & ((1u << lane) - 1u));
                            // footprint centre and half-axes in grid-cell coordinates
                            const float ccx = ffm(A00, x[j], ffm(A01, y[j], gfx));
                            const float ccy = ffm(A10, x[j], ffm(A11, y[j], gfy));
                            const float lx = fm(cs[j], al), ly = fm(sn[j], al);    // body x axis * extent
                            const float wx = fm(-sn[j], hw), wy = fm(cs[j], hw);   // body y axis * hw
                            sts128(pl + 32 * r, make_float4(ccx, ccy, fa(fm(A00, lx), fm(A01, ly)),
                                                            fa(fm(A10, lx), fm(A11, ly))));
                            sts128(pl + 32 * r + 16, make_float4(fa(fm(A00, wx), fm(A01, wy)),
                                                                 fa(fm(A10, wx), fm(A11, wy)), 0.0f, 0.0f));
                        }
                        rank0 += __popc(nm[j]);
                    }
                    __syncwarp();
                    if (discs) {
                        // the three discs of every listed footprint: centre and +- L/3 along the
                        // body axis, one distance-transform lookup each (out of bounds = collision)
                        const int nwork = total * 3;
                        for (int w = lane; w < nwork; w += 32) {
                            const int fp = w / 3;
                            const float sa = (float)(w - 3 * fp) - 1.0f;
                            const float4 P0 = lds128(pl + 32 * fp);
                            const int col = gix + __float2int_rd(fa(P0.x, fm(sa, P0.z)));
                            const int row = giy + __float2int_rd(fa(P0.y, fm(sa, P0.w)));
                            if ((unsigned)col >= (unsigned)gw || (unsigned)row >= (unsigned)gh) hit_map = true;
                            else if ((int)__ldg(a.grid.edt2 + (size_t)row * gw + col) < a.grid.disc_t2) hit_map = true;
                        }
                    } else {
                        // 4 corners, 4 edge mid-points, centre (SURVEY B.6, P = 9): probe p sits at
                        // centre + sa * l-axis + sb * w-axis with (sa, sb) in {-1, 0, 1}, two bits each.
                        // x + (+-1) * e and x + 0 * e round like x +- e and x, so the cells are the
                        // ones the oracle's float32 mirror visits.
                        const int nwork = total * 9;
                        for (int w = lane; w < nwork; w += 32) {
                            const int fp = w / 9, p = w - 9 * fp;
                            const float4 P0 = lds128(pl + 32 * fp), P1 = lds128(pl + 32 * fp + 16);
                            const float sa = (float)(int)((0x1520au >> (2 * p)) & 3u) - 1.0f;
                            const float sb = (float)(int)((0x12522u >> (2 * p)) & 3u) - 1.0f;
                            hit_map |= grid_hit(occ, gw, gh, gix, giy, fa(fa(P0.x, fm(sa, P0.z)), fm(sb, P1.x)),
                                                fa(fa(P0.y, fm(sa, P0.w)), fm(sb, P1.y)));
                        }
                    }
                    __syncwarp();
                }
            }
            if (use_prev) t_sim = warp_sum(sim);
            hit_opp = __any_sync(F1L_FULL, hit_opp);
            hit_map = __any_sync(F1L_FULL, hit_map);
            if (hit_opp) flags |= F1L_FLAG_COLLIDE_OPP;
            if (hit_map) flags |= F1L_FLAG_COLLIDE_MAP;
            if constexpr (PW) {
                partial = partial + lds32(cbase + L::C_GRID + 60) * t_sim;
                if (lane == 0 && a.terms) a.terms[cand * F1L_N_TERMS + 3] = t_sim;
            } else {
                partial = a.ep.w[0] * t_len + a.ep.w[1] * t_maxk + a.ep.w[2] * t_meank + a.ep.w[3] * t_sim;
                if (lane == 0 && a.terms) {
                    float* t = a.terms + cand * F1L_N_TERMS;
                    t[0] = t_len; t[1] = t_maxk; t[2] = t_meank; t[3] = t_sim;
                }
            }

            // ---- raceline deviation: mean over samples of the nearest distance to the window
            //      (nearest_point semantics, utils.py:53-66).  Lane = (sample group sg, segment
            //      group gg); each lane keeps S samples in registers and walks every GG-th
            //      segment, the next segment's table entry already in flight.
            __syncwarp();
            {
                // samples are processed in pairs with packed FP32x2 instructions (FFMA2 / FMUL2,
                // sm_100): the same FMA-pipe work in half the issue slots -- the loop is issue-bound
                // otherwise (1 warp-instruction per clock per scheduler, 9 per sample x segment).
                constexpr int SP = S / 2;
                constexpr bool ODD = (S & 1) != 0;
                f32x2 sx2[SP], sy2[SP];
                float bdx[SP], bdy[SP];
                float sxl = 0.0f, syl = 0.0f, bdl = CUDART_INF_F;
                const uint32_t ra = wbase + L::W_SLABX + sgi * 8;
#pragma unroll
                for (int j = 0; j < SP; ++j) {
                    sx2[j] = lds64(ra + j * SG * 8);
                    sy2[j] = lds64(ra + SLAB * 4 + j * SG * 8);
                    bdx[j] = CUDART_INF_F;
                    bdy[j] = CUDART_INF_F;
                }
                // Odd S: the last sample row is unpacked.  When it holds at most SG / 2 samples
                // (M = 100: 4 of 8, M = 200: 8 of 16) the lanes of the upper half of the sample
                // groups would only carry dummies; instead both halves take the SAME samples and
                // split the two segments of a trip between them -- the lower half tests segment A,
                // the upper half segment B, each from its own table address (one extra LDS.128
                // pair per trip instead of a second 7-instruction scalar chain), and the two
                // halves' minima meet in one shuffle after the loop.
                const bool split_odd = ODD && (M - (S - 1) * SG) <= SG / 2;   // uniform
                if (ODD) {
                    const uint32_t ro = split_odd ? wbase + L::W_SLABX + (sgi & (SG / 2 - 1)) * 8 : ra;
                    sxl = lds32(ro + SP * SG * 8);
                    syl = lds32(ro + SLAB * 4 + SP * SG * 8);
                }
                const int nq = a.nseg_pad;
                // segment range [k_begin, k_end) of the window this candidate is tested against
                int k_begin = 0, k_end = nq;
                if (a.ep.prune && !a.terms && (flags & (F1L_FLAG_COLLIDE_OPP | F1L_FLAG_COLLIDE_MAP))) {
                    // prune mode also drops the scan for a candidate that collided when nobody
                    // asked for its per-term costs: its cost is +inf whatever the deviation
                    k_end = 0;
                } else if (a.ep.prune) {
                    // Every point of a curve of length s_f from the origin to (ex, ey) lies
                    // within rho = s_f / 2 of the chord midpoint c.  With D = the distance of c
                    // to the window, every sample's nearest distance is <= D + rho, and a
                    // segment farther than D + 2 rho from c is farther than D + rho from every
                    // sample: it cannot hold any sample's minimum.  Dropping it leaves every
                    // per-sample minimum, hence the cost, bit-identical.  The kept segments are
                    // covered by one index range (the raceline is a curve: normally one run).
                    const float cmx = 0.5f * ex * EVAL_DEV_SCALE, cmy = 0.5f * ey * EVAL_DEV_SCALE;
                    const uint32_t tb = cbase + L::C_TAB;
                    float dmin = CUDART_INF_F;
                    for (int k = lane; k < nq; k += 32)
                        dmin = fminf(dmin, seg_dist2(cmx, cmy, lds128(tb + 32 * k), lds128(tb + 32 * k + 16)));
                    dmin = __uint_as_float(__reduce_min_sync(F1L_FULL, __float_as_uint(dmin)));
                    // 1 mm + 0.1 % of slack over the rounding of the FP32 distances and samples
                    const float thr = (fast_sqrt(dmin) + sp.sf * EVAL_DEV_SCALE) * 1.001f + 1e-3f * EVAL_DEV_SCALE;
                    const float thr2 = thr * thr;
                    int lo = nq, hi = -1;
                    for (int k = lane; k < nq; k += 32)
                        if (seg_dist2(cmx, cmy, lds128(tb + 32 * k), lds128(tb + 32 * k + 16)) <= thr2) {
                            lo = min(lo, k);
                            hi = max(hi, k);
                        }
                    lo = __reduce_min_sync(F1L_FULL, lo);
                    hi = __reduce_max_sync(F1L_FULL, hi);
                    if (hi >= lo) {   // (always: the nearest segment itself passes)
                        k_begin = lo & ~(2 * GG - 1);
                        k_end = min(nq, (hi + 2 * GG) & ~(2 * GG - 1));
                    }
                }
                if (a.stats && lane == 0 && k_end > k_begin) atomicAdd(&s_work, (1ull << 40) + (unsigned long long)(k_end - k_begin));
                // the walk advances the table address itself (one add per trip); the trip count is
                // warp-uniform and lives in a uniform register
                uint32_t ta = cbase + L::C_TAB + (k_begin + ggi) * 32;
                float4 T0 = lds128(ta), T1 = lds128(ta + 16);
                // two segments per trip: the running minimum takes both distances in one
                // three-input FMNMX3 (nseg_pad / GG is a multiple of 8).  The next trip's entries
                // are loaded at the end of the trip (fewer live registers than a prefetch into
                // registers at its start, measured faster).
                if (split_odd) {
                    const uint32_t off = (sgi >= SG / 2) ? GG * 32 : 0;   // this lane's segment of the trip
                    for (int n = (k_end - k_begin) / (2 * GG); n > 0; --n) {
                        const float4 B0 = lds128(ta + GG * 32), B1 = lds128(ta + GG * 32 + 16);
                        seg_min2<SP>(sx2, sy2, T0, T1, B0, B1, bdx, bdy);
                        const uint32_t to = ta + off;
                        bdl = fminf(bdl, seg_dist2(sxl, syl, lds128(to), lds128(to + 16)));
                        ta += 2 * GG * 32;
                        T0 = lds128(ta);   // EVAL_SEG_PAD entries of slack
                        T1 = lds128(ta + 16);
                    }
                    bdl = fminf(bdl, __shfl_xor_sync(F1L_FULL, bdl, (SG / 2) * GG));
                } else {
                    for (int n = (k_end - k_begin) / (2 * GG); n > 0; --n) {
                        const float4 B0 = lds128(ta + GG * 32), B1 = lds128(ta + GG * 32 + 16);
                        seg_min2<SP>(sx2, sy2, T0, T1, B0, B1, bdx, bdy);
                        if (ODD) bdl = fmin3(bdl, seg_dist2(sxl, syl, T0, T1), seg_dist2(sxl, syl, B0, B1));
                        ta += 2 * GG * 32;
                        T0 = lds128(ta);   // EVAL_SEG_PAD entries of slack
                        T1 = lds128(ta + 16);
                    }
                }
                // Minima over the GG lanes of a sample group, by halving: at every step a lane keeps
                // one half of its rows and hands the other half to its partner, so it ends with S / GG
                // fully reduced rows of its own (7 + 4 shuffles and 4 square roots for S = 13, GG = 4,
                // against 26 shuffles and 13 square roots on every lane when all lanes reduce all rows).
                float rows[S];
#pragma unroll
                for (int j = 0; j < SP; ++j) { rows[2 * j] = bdx[j]; rows[2 * j + 1] = bdy[j]; }
                if (ODD) rows[S - 1] = bdl;
                const float dsum = halve_min_sqrt_sum<S, GG>(rows, ggi, nrows);
                t_dev = warp_sum(dsum) * ((1.0f / EVAL_DEV_SCALE) * a.ep.inv_M);
            }

            if (!(flags & (F1L_FLAG_COLLIDE_OPP | F1L_FLAG_COLLIDE_MAP))) {
                cost = partial + (PW ? lds32(cbase + L::C_GRID + 44) : a.ep.w[4]) * t_dev;
                if (!isfinite(cost)) cost = CUDART_INF_F;
            }
        }

        if (lane == 0) {
            if (a.costs) a.costs[cand] = cost;
            if (a.flags) a.flags[cand] = (uint8_t)flags;
            if (a.terms) {
                float* t = a.terms + cand * F1L_N_TERMS;
                if (!(flags & F1L_FLAG_VALID)) { t[0] = 0.0f; t[1] = 0.0f; t[2] = 0.0f; t[3] = 0.0f; }
                t[4] = t_dev;
            }
            const unsigned long long key =
                ((unsigned long long)float_orderable(cost) << 32) | (unsigned)c;
            atomicMin(a.best + s, key);
        }
      }
      __syncwarp();   // all lanes have read the item's solutions
      int c_next = 0;
      if (lane == 0) c_next = dyn ? cb + atomicAdd(a.work_next, item) : atomicAdd(&s_next, item);
      c0 = __shfl_sync(F1L_FULL, c_next, 0);
    }
    if (a.stats) {   // work counters (opt-in, f1l_set_stats): one pair of global atomics per CTA
        __syncthreads();
        if (tid == 0) {
            atomicAdd(a.stats, s_work & ((1ull << 40) - 1));
            atomicAdd(a.stats + 1, s_work >> 40);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K5: select + regenerate + tracker, one warp per scenario
// ---------------------------------------------------------------------------------------------
#define SELECT_THREADS 32
template <int IPL>
__global__ void __launch_bounds__(SELECT_THREADS) select_kernel(SelectArgs a) {
    __shared__ float4 s_traj[F1L_MAX_M];
    const int s = blockIdx.x, lane = threadIdx.x;
    const int M = a.ep.M;
    const QueryCtx* __restrict__ q = a.ctx + s;
    unsigned long long key = a.best[s];
    // goal centre of the winner's lookahead row.  A shard's sampler fills only the rows the shard
    // evaluates, which contain its own winner; in a sharded query the global winner's centre
    // arrives with its key through the exchange.
    Centre ce;
    ce.cx = 0.f; ce.cy = 0.f; ce.psi_rel = 0.f; ce.kappa_g = 0.f; ce.nx = 0.f; ce.ny = 0.f; ce.v = 0.f; ce.ok = 0.f;
    if (!a.goals) {
        const int lidx = key == ~0ull ? a.c_begin : (int)(key & 0xffffffffu);
        const int lrow = __float2int_rd(((float)lidx + 0.5f) * a.inv_nW);
        const int rel = lrow - a.row0;
        if (rel >= 0 && rel < a.n_rows * a.row_step && (a.row_step == 1 || rel % a.row_step == 0))
            ce = a.centres[(size_t)s * a.nL + lrow];   // (a rank without rows has nothing to offer)
    }
    if (a.xc.world > 1) {   // (S == 1) the ranks' local minima meet over NVLink peer memory
        int timed_out = 0;
        key = xchg_global_min(a.xc, key, ce, lane, &timed_out);
        if (lane == 0 && a.xchg_status) *a.xchg_status = timed_out;
    }
    int idx = (int)(key & 0xffffffffu);
    float cost = orderable_float((uint32_t)(key >> 32));
    const bool none = (key == ~0ull) || !(cost < CUDART_INF_F);
    if (key == ~0ull) { idx = a.c_begin; cost = CUDART_INF_F; }

    float gx, gy, gth, p3, v_ref;
    bool have_centre;
    // speed column / tracker speed: the raceline speed at the goal centre, read back in float64
    // from the waypoint the sampler chose (pure_pursuit.py:78 returns waypoints[i, 2] itself);
    // explicit goals have no centre: the ego speed
    double v_goal = q->vel;
    if (a.goals) {
        candidate_goal(a.centres, a.widths, a.goals, a.nL, a.nW, a.inv_nW, a.C, s, idx,
                       a.ep.use_goal_kappa != 0, gx, gy, gth, p3, have_centre, v_ref);
    } else {
        const int row = __float2int_rd(((float)idx + 0.5f) * a.inv_nW), k = idx - row * a.nW;
        const float wk = __ldg(a.widths + k);
        gx = fmaf(wk, ce.nx, ce.cx);
        gy = fmaf(wk, ce.ny, ce.cy);
        gth = ce.psi_rel;
        p3 = a.ep.use_goal_kappa != 0 ? ce.kappa_g : 0.0f;
        have_centre = ce.ok != 0.0f;
        v_ref = ce.v;
        const int wp = (int)ce.ok - 1;
        if (a.tr.ncols > 2 && wp >= 0) v_goal = a.tr.v[wp];
    }
    SpiralF sp;
    generate_spiral(sp, a.lut, a.ep, gx, gy, gth, p3, lane);
    float x[IPL], y[IPL], th[IPL], kp[IPL], cs[IPL], sn[IPL];
    spiral_sample<IPL>(sp, M, lane, x, y, th, kp, cs, sn);
#pragma unroll
    for (int j = 0; j < IPL; ++j) {
        const int i = lane * IPL + j;
        if (i < M) {
            const float4 st = make_float4(x[j], y[j], th[j], kp[j]);
            s_traj[i] = st;
            if (a.best_traj) a.best_traj[(size_t)s * M + i] = st;
            if (a.prev_theta_out) a.prev_theta_out[(size_t)s * M + i] = th[j];
        }
    }
    if (a.prev_valid_out && lane == 0) a.prev_valid_out[s] = 1;
    if (a.best_traj_map) {   // warp-uniform
        // map-frame copy with a speed column, what a tracker in the map frame consumes (SURVEY B.8):
        // X = pose + R(theta_pose) (x, y), Theta = theta + theta_pose, v = raceline speed at the
        // goal centre (explicit goals: the ego speed), in float64 from the float32 states
        double sth, cth;
        sincos(q->th, &sth, &cth);
        const double v_col = v_goal;
#pragma unroll
        for (int j = 0; j < IPL; ++j) {
            const int i = lane * IPL + j;
            if (i < M) {
                double* o = a.best_traj_map + 4 * ((size_t)s * M + i);
                const double xd = (double)x[j], yd = (double)y[j];
                o[0] = q->px + (cth * xd - sth * yd);
                o[1] = q->py + (sth * xd + cth * yd);
                o[2] = v_col;
                o[3] = (double)th[j] + q->th;
            }
        }
    }
    __syncwarp();

    // tracker: pure pursuit on the best trajectory (lattice_planner.py:208-212)
    const bool literal = a.ep.literal_tracker != 0;
    const double qx = literal ? q->px : 0.0, qy = literal ? q->py : 0.0;
    const double qth = literal ? q->th : 0.0;
    const double L = a.ep.tracker_lookahead;
    const double wb = literal ? 0.33 : a.ep.wheelbase;  // :55 tracker built with the default
    XYTraj4 acc{s_traj};
    double bd = CUDART_INF;
    int bi = 0x7fffffff;
    {
        // The vehicle-frame tracker queries the trajectory's own first point: segment 0 at
        // distance exactly 0 is the first minimum whatever the other segments give, so the scan
        // is skipped (any other outcome of segment 0 -- the literal mode, a degenerate
        // trajectory -- takes the full scan).
        const double2 p0 = acc(0), p1 = acc(1);
        double ux, uy, d, t;
        nearest_segment64(qx, qy, p0.x, p0.y, p1.x, p1.y, ux, uy, d, t);
        if (d == 0.0) { bd = 0.0; bi = 0; }   // warp-uniform
    }
    if (bi != 0) {
        for (int k = lane; k < M - 1; k += 32) {
            const double2 p0 = acc(k), p1 = acc(k + 1);
            double ux, uy, d, t;
            nearest_segment64(qx, qy, p0.x, p0.y, p1.x, p1.y, ux, uy, d, t);
            // NaN distances (degenerate trajectory) never win; the reference would return them
            if (nearest_better(d, k, bd, bi)) { bd = d; bi = k; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(F1L_FULL, bd, o);
            const int oi = __shfl_xor_sync(F1L_FULL, bi, o);
            if (nearest_better(od, oi, bd, bi)) { bd = od; bi = oi; }
        }
    }
    int found = 0;
    double steer = 0.0, speed = 0.0;
    if (bi != 0x7fffffff) {   // warp-uniform
        const double2 p0 = acc(bi), p1 = acc(bi + 1);
        double ux, uy, d, t;
        nearest_segment64(qx, qy, p0.x, p0.y, p1.x, p1.y, ux, uy, d, t);
        const double v_track = literal ? (double)s_traj[bi].z : v_goal;
        double lx = 0.0, ly = 0.0;
        if (d < L) {                                        // pure_pursuit.py:70
            const Intersect64 ip = intersect_point_warp(acc, M, qx, qy, L, (double)bi + t, true,
                                                        lane, NoPrefilter());
            if (ip.found) {
                const int r = pymod(ip.i, M);
                lx = acc(r).x; ly = acc(r).y;
                found = 1;
            }
        } else if (d < a.ep.max_reacquire) {                 // :80
            lx = p0.x; ly = p0.y;
            found = 1;
        }
        if (found) {
            steer = actuation_steer64(qth, lx, ly, qx, qy, L, wb);
            speed = v_track;
        }
    }
    if (lane == 0) {
        if (a.best_idx) a.best_idx[s] = idx;
        if (a.best_cost) a.best_cost[s] = cost;
        if (a.status) { a.status[2 * s] = none ? 1 : 0; a.status[2 * s + 1] = found; }
        if (a.steer_speed) { a.steer_speed[2 * (size_t)s] = steer; a.steer_speed[2 * (size_t)s + 1] = speed; }
    }
}

// Chebyshev clearance of every cell (distance in cells to the nearest occupied or out-of-bounds
// cell, capped at R+1), separable: horizontal pass then vertical pass.
#define CLEAR_R 24
__global__ void clearance_h_kernel(const uint8_t* __restrict__ occ, int h, int w,
                                   uint8_t* __restrict__ hd) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
    if (col >= w) return;
    const uint8_t* r = occ + (size_t)row * w;
    int d = CLEAR_R + 1;
    if (r[col]) d = 0;
    else
        for (int k = 1; k <= CLEAR_R; ++k) {
            const int a = col - k, b = col + k;
            if (a < 0 || b >= w || r[a] || r[b]) { d = k; break; }
        }
    hd[(size_t)row * w + col] = (uint8_t)d;
}
__global__ void clearance_v_kernel(const uint8_t* __restrict__ hd, int h, int w,
                                   uint16_t* __restrict__ clear) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
    if (col >= w) return;
    int best = hd[(size_t)row * w + col];
    for (int k = 1; k <= CLEAR_R && k < best; ++k) {
        const int a = row - k, b = row + k;
        int da = 0, db = 0;
        if (a >= 0) da = hd[(size_t)a * w + col];
        if (b < h) db = hd[(size_t)b * w + col];
        const int m = max(k, min(da, db));
        best = min(best, m);
    }
    clear[(size_t)row * w + col] = (uint16_t)best;
}

// Exact Euclidean distance transform up to CLEAR_R cells, second (vertical) pass over the
// horizontal distances `hd` of clearance_h_kernel (0 = occupied, out of bounds counts as
// occupied, CLEAR_R + 1 = farther):  d^2(r, c) = min over dr of dr^2 + hd(r + dr, c)^2.  A nearest
// occupied cell within Euclidean distance CLEAR_R has |dr|, |dc| <= CLEAR_R, so every value up to
// CLEAR_R^2 is exact; larger ones are stored as the sentinel CLEAR_R^2 + 1.
#define EDT_FAR (CLEAR_R * CLEAR_R + 1)
__global__ void edt_v_kernel(const uint8_t* __restrict__ hd, int h, int w, uint16_t* __restrict__ edt2) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
    if (col >= w) return;
    int best = EDT_FAR;
    for (int dr = -CLEAR_R; dr <= CLEAR_R; ++dr) {
        const int r = row + dr;
        int d = 0;                                            // a row outside the grid is occupied
        if (r >= 0 && r < h) d = hd[(size_t)r * w + col];
        if (d > CLEAR_R) continue;                            // nothing within reach in that row
        best = min(best, dr * dr + d * d);
    }
    edt2[(size_t)row * w + col] = (uint16_t)min(best, EDT_FAR);
}

__global__ void fill_f32_kernel(float* __restrict__ p, size_t n, float v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------------------------
// generate-only kernel (user cost functions on the host): goals -> states / params / flags
// ---------------------------------------------------------------------------------------------
template <int IPL>
__global__ void __launch_bounds__(EVAL_MAX_WARPS * 32)
generate_kernel(LutView lut, EvalParams ep, const float4* __restrict__ goals, int C,
                float4* __restrict__ states, float4* __restrict__ params,
                uint8_t* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= C) return;
    const int M = ep.M;
    const float4 g = __ldg(goals + c);
    SpiralF sp;
    generate_spiral(sp, lut, ep, g.x, g.y, g.z, g.w, lane);
    float x[IPL], y[IPL], th[IPL], kp[IPL], cs[IPL], sn[IPL];
    spiral_sample<IPL>(sp, M, lane, x, y, th, kp, cs, sn);
    float maxk = 0.0f, ex = 0.0f, ey = 0.0f, eth = 0.0f;
#pragma unroll
    for (int j = 0; j < IPL; ++j) {
        const int i = lane * IPL + j;
        if (i < M) {
            states[(size_t)c * M + i] = make_float4(x[j], y[j], th[j], kp[j]);
            maxk = fmaxf(maxk, fabsf(kp[j]));
            if (i == M - 1) { ex = x[j]; ey = y[j]; eth = th[j]; }
        }
    }
    const int last_lane = (M - 1) / IPL;
    ex = __shfl_sync(F1L_FULL, ex, last_lane);
    ey = __shfl_sync(F1L_FULL, ey, last_lane);
    eth = __shfl_sync(F1L_FULL, eth, last_lane);
    maxk = warp_max(maxk);
    const float gn = sqrtf(fmaf(g.x, g.x, fmaf(g.y, g.y, g.z * g.z)));
    const float tol = ep.tol * fmaxf(gn, 1.0f);
    bool valid = isfinite(sp.p1) && isfinite(sp.p2) && isfinite(sp.sf) && sp.sf > 0.0f &&
                 fabsf(ex - g.x) < tol && fabsf(ey - g.y) < tol && fabsf(eth - g.z) < tol;
    if (valid && ep.kappa_max > 0.0f && !(maxk <= ep.kappa_max)) valid = false;
    if (lane == 0) {
        if (params)
            params[c] = ep.generator == 1 ? make_float4(sp.p0, __fdividef(sp.b1, sp.sf), sp.sf, sp.p3)
                                          : make_float4(sp.p1, sp.p2, sp.sf, sp.p3);
        if (flags) flags[c] = valid ? F1L_FLAG_VALID : 0;
    }
}

// ---------------------------------------------------------------------------------------------
// spiral seed LUT build, float64, one thread per cell (SURVEY B.2: continuation from the
// straight line to the cell's goal, then polishing; non-converged cells get the heuristic seed)
// ---------------------------------------------------------------------------------------------
__device__ inline bool newton_step64(double gx, double gy, double gth, double& p1, double& p2,
                                     double& sf) {
    const double b1 = (18.0 * p1 - 9.0 * p2) / 2.0;
    const double b2 = (-45.0 * p1 + 36.0 * p2) / 2.0;
    const double b3 = (27.0 * p1 - 27.0 * p2) / 2.0;
    double C0 = 0, S0 = 0, Cg = 0, Sg = 0, C1 = 0, S1 = 0, C2 = 0, S2 = 0;
    for (int j = 0; j <= 32; ++j) {
        const double u = (double)j / 32.0;
        const double w = ((j == 0 || j == 32) ? 1.0 : ((j & 1) ? 4.0 : 2.0)) / 96.0;
        const double g = u * (u * (b1 / 2.0 + u * (b2 / 3.0 + u * (b3 / 4.0))));
        const double th = sf * g;
        const double c = cos(th), s = sin(th);
        const double u2 = u * u;
        const double d1 = u2 * (4.5 + u * (-7.5 + 3.375 * u));
        const double d2 = u2 * (-2.25 + u * (6.0 - 3.375 * u));
        C0 += w * c; S0 += w * s; Cg += w * c * g; Sg += w * s * g;
        C1 += w * c * d1; S1 += w * s * d1; C2 += w * c * d2; S2 += w * s * d2;
    }
    const double g1 = (3.0 * p1 + 3.0 * p2) / 8.0;
    const double r0 = sf * C0 - gx, r1 = sf * S0 - gy, r2 = sf * g1 - gth;
    const double sf2 = sf * sf;
    const double J00 = -sf2 * S1, J01 = -sf2 * S2, J02 = C0 - sf * Sg;
    const double J10 = sf2 * C1, J11 = sf2 * C2, J12 = S0 + sf * Cg;
    const double J20 = 0.375 * sf, J21 = 0.375 * sf, J22 = g1;
    const double m0 = J11 * J22 - J12 * J21, m1 = J10 * J22 - J12 * J20, m2 = J10 * J21 - J11 * J20;
    const double det = J00 * m0 - J01 * m1 + J02 * m2;
    const double inv = 1.0 / det;
    const double n0 = r1 * J22 - J12 * r2, n1 = r1 * J21 - J11 * r2, n2 = J10 * r2 - r1 * J20;
    p1 -= (r0 * m0 - J01 * n0 + J02 * n1) * inv;
    p2 -= (J00 * n0 - r0 * m1 + J02 * n2) * inv;
    sf -= (-J00 * n1 - J01 * n2 + r0 * m2) * inv;
    return isfinite(p1) && isfinite(p2) && isfinite(sf);
}

__device__ inline double residual64(double gx, double gy, double gth, double p1, double p2,
                                    double sf) {
    const double b1 = (18.0 * p1 - 9.0 * p2) / 2.0;
    const double b2 = (-45.0 * p1 + 36.0 * p2) / 2.0;
    const double b3 = (27.0 * p1 - 27.0 * p2) / 2.0;
    double C0 = 0, S0 = 0;
    for (int j = 0; j <= 32; ++j) {
        const double u = (double)j / 32.0;
        const double w = ((j == 0 || j == 32) ? 1.0 : ((j & 1) ? 4.0 : 2.0)) / 96.0;
        const double th = sf * (u * (u * (b1 / 2.0 + u * (b2 / 3.0 + u * (b3 / 4.0)))));
        C0 += w * cos(th); S0 += w * sin(th);
    }
    const double g1 = (3.0 * p1 + 3.0 * p2) / 8.0;
    return fmax(fabs(sf * C0 - gx), fmax(fabs(sf * S0 - gy), fabs(sf * g1 - gth)));
}

__global__ void lut_build_kernel(float4* __restrict__ cells, int nx, int ny, int nt, double x0,
                                 double x1, double y0, double y1, double t0, double t1) {
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= nx * ny * nt) return;
    const int it = cell % nt, iy = (cell / nt) % ny, ix = cell / (nt * ny);
    const double gx = nx > 1 ? x0 + (x1 - x0) * (double)ix / (double)(nx - 1) : x0;
    const double gy = ny > 1 ? y0 + (y1 - y0) * (double)iy / (double)(ny - 1) : y0;
    const double gt = nt > 1 ? t0 + (t1 - t0) * (double)it / (double)(nt - 1) : t0;
    double p1 = 0.0, p2 = 0.0, sf = gx;
    bool ok = gx > 0.0;
    for (int s = 1; s <= 16 && ok; ++s) {
        const double lam = (double)s / 16.0;
        for (int k = 0; k < 4 && ok; ++k) ok = newton_step64(gx, lam * gy, lam * gt, p1, p2, sf);
        if (!(sf > 0.0)) ok = false;
    }
    for (int k = 0; k < 8 && ok; ++k) ok = newton_step64(gx, gy, gt, p1, p2, sf);
    if (ok && sf > 0.0 && residual64(gx, gy, gt, p1, p2, sf) < 1e-8) {
        cells[cell] = make_float4((float)p1, (float)p2, (float)sf, 1.0f);
    } else {
        const double d = sqrt(gx * gx + gy * gy);
        cells[cell] = make_float4(0.0f, 0.0f, (float)(d * (gt * gt / 5.0 + 1.0) + 2.0 * fabs(gt) / 5.0),
                                  0.0f);
    }
}
