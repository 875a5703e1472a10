// f1l_common.cuh -- shared device structs and helpers for the sm_100a lattice-planner kernels.
//
// Reference citations are into f1tenth_planning/ of the upstream repo.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/f1l.h"

#define F1L_WARP 32
#define F1L_FULL 0xffffffffu
#define F1L_MAX_LOOKAHEADS 1024

// ---------------------------------------------------------------------------------------------
// device-side views
// ---------------------------------------------------------------------------------------------
struct TrackView {
    int n;                 // waypoints
    int ncols;             // columns uploaded (2..5)
    const double2* xy;     // [n] map frame, float64 (exact copy of the host array)
    const double* v;       // [n] column 2 (speed) or zeros
    const double* psi;     // [n] column 3 or zeros
    const double* kappa;   // [n] column 4 or zeros
    // float32 line form of the n-1 open segments in block-local frames (nearest-point scans), in
    // table units of TRACK_UNIT metres (see track_seg_d2):
    //   segA[k] = (ux, uy, -(a.u + h), -a.n): unit direction u, normal n = (-uy, ux), a = segment
    //   start relative to the origin of block k/32, h = len / 2;  segB[k] = (-h, -uy)
    const float4* segA;
    const float2* segB;
    const double2* blk_origin;  // [ceil((n-1)/32)]
};

struct GridView {
    const uint8_t* occ;    // [h, w] row-major, 0 free
    // [h, w] uint16 "how far is the nearest occupied / out-of-bounds cell" map the footprint test
    // looks up first (or null): collision_mode 0 -- Chebyshev clearance in cells (0 = occupied);
    // collision_mode 1 -- squared Euclidean cell distance (edt2).  A sample whose value is at least
    // near_free cannot collide and skips the per-footprint test.
    const uint16_t* near_map;
    int near_free;
    int h, w;
    double ox, oy, inv_res;
    // collision_mode 1: three discs on the Euclidean distance transform
    const uint16_t* edt2;  // [h, w] squared cell distance to the nearest occupied / out-of-bounds cell
    int disc_t2;           // a disc collides iff edt2[its centre's cell] < disc_t2 = ceil((r_disc / res)^2)
    float disc_off;        // disc spacing along the body axis, L / 3 (metres)
};

struct LutView {
    const float4* cells;  // [nx, ny, nt] (p1, p2, s_f, converged)
    int nx, ny, nt;
    float x0, y0, t0;     // axis origins
    float sx, sy, st;     // (n-1)/(hi-lo) per axis (0 when n == 1)
};

// planner constants in the types the kernels use
struct EvalParams {
    int M;            // arc samples
    int n_newton;
    int window;       // requested window (<=0: all)
    int n_shift, n_cull;
    int literal_tracker, use_goal_kappa;
    int generator;    // 0 cubic spiral, 1 G1 clothoid
    int prune;        // deviation pass: skip window segments that cannot be nearest
    int collision_mode;  // 0 nine probes, 1 three discs on the distance transform
    float w[F1L_N_TERMS];
    float kappa_max;  // <= 0: off
    float half_l, half_w;
    float rc2;        // (2 r_circ)^2 broad-phase radius
    float reach_pad;  // 2 r_circ + 1 mm: candidate-level opponent prune
    float inv_M;      // 1 / M
    float tol;
    double tracker_lookahead, wheelbase, max_reacquire;
};

// per-scenario context written by the sampler kernel, read by eval / select
struct __align__(16) QueryCtx {
    double px, py, th, vel;
    double t_ego;          // parameter of the nearest point on segment i_ego (utils.py:58-60)
    double pad1;
    float cth, sth;        // cos / sin of the pose heading
    int i_ego;             // nearest open-polyline segment (utils.py:66)
    int seg0, nseg;        // cyclic raceline window [seg0, seg0+nseg) over the n-1 segments
    int n_opp;
    int has_grid;
    int pad0;
    // vehicle frame -> grid cell coordinates: cell = i0 + floor(A * (x, y) + f)
    float gA00, gA01, gA10, gA11, gfx, gfy;
    int gix, giy;
    float4 opp[F1L_MAX_OPP];  // vehicle frame (x, y, cos phi, sin phi)
};

// per lookahead row: goal centre in the vehicle frame
struct __align__(16) Centre {
    float cx, cy, psi_rel, kappa_g;  // centre xy, wrap(psi - theta), raceline curvature
    float nx, ny, v, ok;             // unit normal (-sin psi_rel, cos psi_rel), raceline speed, found
};

// FP32 squared distance (table units squared) of a block-relative point, already in table units,
// to segment k of the uploaded line form: q_c = p.u - (a.u + h) is the coordinate along the
// segment measured from its midpoint, so the excess beyond the segment is max(|q_c| - h, 0) =
// sat(|q_c| - h) -- one FADD.SAT with an |.| operand modifier -- as long as it stays below one
// table unit, which TRACK_UNIT = 16384 m guarantees for any real track.  7 FMA-pipe instructions.
#define TRACK_UNIT 16384.0f
#define TRACK_SCALE (1.0f / TRACK_UNIT)
__device__ __forceinline__ float track_seg_d2(float prx, float pry, float4 A, float2 Bv) {
    const float q = fmaf(prx, A.x, fmaf(pry, A.y, A.z));
    const float nn = fmaf(pry, A.x, fmaf(-prx, A.y, A.w));
    const float e = __saturatef(fabsf(q) + Bv.x);
    return fmaf(e, e, nn * nn);
}

// ---------------------------------------------------------------------------------------------
// float64 helpers that follow the reference operation by operation (no FMA contraction)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double xmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xsub(double a, double b) { return __dsub_rn(a, b); }

struct Nearest64 {
    double px, py, dist, t;
    int i;
};

// one segment of nearest_point (utils/utils.py:53-65)
__device__ __forceinline__ void nearest_segment64(double qx, double qy, double ax, double ay,
                                                  double bx, double by, double& px, double& py,
                                                  double& dist, double& t) {
    const double dx = xsub(bx, ax), dy = xsub(by, ay);                       // :53
    const double l2 = xadd(xmul(dx, dx), xmul(dy, dy));                       // :54
    const double dot = xadd(xmul(xsub(qx, ax), dx), xmul(xsub(qy, ay), dy));  // :57
    double tt = __ddiv_rn(dot, l2);                                           // :58
    if (tt < 0.0) tt = 0.0;                                                   // :59
    if (tt > 1.0) tt = 1.0;                                                   // :60
    px = xadd(ax, xmul(tt, dx));                                              // :61
    py = xadd(ay, xmul(tt, dy));
    const double ex = xsub(qx, px), ey = xsub(qy, py);                        // :64
    dist = __dsqrt_rn(xadd(xmul(ex, ex), xmul(ey, ey)));                      // :65
    t = tt;
}

// float64 re-evaluation of an FP32 argmin: segments [k-2, k+2], first minimum (utils.py:66)
__device__ __forceinline__ Nearest64 refine_nearest64(const double2* __restrict__ xy, int nseg,
                                                      double qx, double qy, int k) {
    Nearest64 b;
    b.dist = CUDART_INF; b.i = 0; b.px = 0.0; b.py = 0.0; b.t = 0.0;
    const int lo = max(k - 2, 0), hi = min(k + 2, nseg - 1);
    // the five evaluations are independent (a division and a square root each): computed side by
    // side, then the first-minimum rule replayed in segment order
    double px[5], py[5], d[5], t[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const int s = min(lo + j, hi);   // (slots beyond hi repeat the last segment and are not used)
        const double2 a = xy[s], c = xy[s + 1];
        nearest_segment64(qx, qy, a.x, a.y, c.x, c.y, px[j], py[j], d[j], t[j]);
    }
#pragma unroll
    for (int j = 0; j < 5; ++j)
        if (lo + j <= hi && d[j] < b.dist) { b.dist = d[j]; b.i = lo + j; b.px = px[j]; b.py = py[j]; b.t = t[j]; }
    return b;
}

// The same with the (up to) five segments on five lanes of a converged warp: one float64 segment
// evaluation deep instead of five; the first-minimum rule is replayed in segment order over the
// shuffled distances.  Every lane returns the result.
__device__ __forceinline__ Nearest64 refine_nearest64_warp(const double2* __restrict__ xy, int nseg,
                                                           double qx, double qy, int k, int lane) {
    const int lo = max(k - 2, 0), hi = min(k + 2, nseg - 1);
    const int s = lo + lane;
    double px = 0.0, py = 0.0, d = CUDART_INF, t = 0.0;
    if (s <= hi) {
        const double2 a = xy[s], c = xy[s + 1];
        nearest_segment64(qx, qy, a.x, a.y, c.x, c.y, px, py, d, t);
    }
    double bd = CUDART_INF;
    int bj = -1;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const double dj = __shfl_sync(0xffffffffu, d, j);
        if (lo + j <= hi && dj < bd) { bd = dj; bj = j; }
    }
    Nearest64 b;
    b.dist = CUDART_INF; b.i = 0; b.px = 0.0; b.py = 0.0; b.t = 0.0;
    const int src = bj < 0 ? 0 : bj;
    const double wpx = __shfl_sync(0xffffffffu, px, src), wpy = __shfl_sync(0xffffffffu, py, src);
    const double wt = __shfl_sync(0xffffffffu, t, src);
    if (bj >= 0) { b.dist = bd; b.i = lo + bj; b.px = wpx; b.py = wpy; b.t = wt; }
    return b;
}

// lexicographic (dist, index) minimum == np.argmin first-minimum rule (utils.py:66)
__device__ __forceinline__ bool nearest_better(double d, int i, double bd, int bi) {
    return d < bd || (d == bd && i < bi);
}

// python-style modulo for the index range the scans use (-n <= a < 2n): no integer division
__device__ __forceinline__ int pymod(int a, int n) {
    if (a < 0) a += n;
    else if (a >= n) a -= n;
    return a;
}

// accessor concept: P(i) returns double2 waypoint i
struct XYTrack {
    const double2* xy;
    __device__ __forceinline__ double2 operator()(int i) const { return xy[i]; }
};
struct XYTraj4 {  // float4 trajectory rows (x, y, theta, kappa) widened to float64
    const float4* st;
    __device__ __forceinline__ double2 operator()(int i) const {
        const float4 s = st[i];
        return make_double2((double)s.x, (double)s.y);
    }
};

// one segment test of intersect_point (utils/utils.py:85-101); returns false if disc < 0
__device__ __forceinline__ bool intersect_segment64(double qx, double qy, double r, double2 s,
                                                    double2 e0, double& t1, double& t2,
                                                    double& vx, double& vy) {
    const double ex = xadd(e0.x, 1e-6), ey = xadd(e0.y, 1e-6);  // :86
    vx = xsub(ex, s.x);
    vy = xsub(ey, s.y);
    const double a = xadd(xmul(vx, vx), xmul(vy, vy));                                  // :89
    const double b = xmul(2.0, xadd(xmul(vx, xsub(s.x, qx)), xmul(vy, xsub(s.y, qy))));  // :90
    const double c = xsub(xsub(xadd(xadd(xmul(s.x, s.x), xmul(s.y, s.y)),
                                    xadd(xmul(qx, qx), xmul(qy, qy))),
                               xmul(2.0, xadd(xmul(s.x, qx), xmul(s.y, qy)))),
                          xmul(r, r));                                                   // :91
    double disc = xsub(xmul(b, b), xmul(xmul(4.0, a), c));                               // :92
    if (disc < 0.0) return false;                                                        // :94
    disc = __dsqrt_rn(disc);
    t1 = __ddiv_rn(xsub(-b, disc), xmul(2.0, a));                                        // :100
    t2 = __ddiv_rn(xadd(-b, disc), xmul(2.0, a));
    return true;
}

struct Intersect64 {
    double px, py, t;
    int i;      // un-modded segment index (may be -1, utils.py:125)
    int found;
};

// prefilter on the uploaded track, FP32 on the block-local line form of segment i.  A root of the
// reference's quadratic in [0,1] is a point of the (1e-6-shifted) segment at distance r from the
// query, so a segment (a) farther than r + 1 mm from the query, or (b) whose FARTHER endpoint is
// closer than r - 2 mm -- the whole segment lies strictly inside the circle -- cannot be accepted
// and needs no float64 test.  (b) is what makes long lookaheads cheap: every segment between the
// query and the crossing is of that kind.  The closing segment (i = -1) has no line form and is
// always tested.
struct TrackPrefilter {
    const TrackView& tr;
    double qx, qy;
    float rr2;   // (radius + 1 mm)^2 in metres^2
    float ri2;   // (max(radius - 2 mm, 0))^2
    __device__ __forceinline__ bool operator()(int i) const {
        if (i < 0) return true;
        const double2 o = tr.blk_origin[i >> 5];
        const float prx = (float)(qx - o.x) * TRACK_SCALE, pry = (float)(qy - o.y) * TRACK_SCALE;
        const float4 A = __ldg(tr.segA + i);
        const float2 Bv = __ldg(tr.segB + i);
        const float q = fmaf(prx, A.x, fmaf(pry, A.y, A.z));
        const float nn = fmaf(pry, A.x, fmaf(-prx, A.y, A.w));
        const float n2 = nn * nn;
        const float e = __saturatef(fabsf(q) + Bv.x);   // beyond the nearer end (Bv.x = -h)
        const float f = fabsf(q) - Bv.x;                // along-axis distance to the farther end
        return fmaf(e, e, n2) <= rr2 * (TRACK_SCALE * TRACK_SCALE) &&
               fmaf(f, f, n2) >= ri2 * (TRACK_SCALE * TRACK_SCALE);
    }
};
__device__ __forceinline__ TrackPrefilter track_prefilter(const TrackView& tr, double qx, double qy, double r) {
    const float ro = (float)r + 1e-3f, ri = fmaxf((float)r - 2e-3f, 0.0f);
    return TrackPrefilter{tr, qx, qy, ro * ro, ri * ri};
}
struct NoPrefilter {
    __device__ __forceinline__ bool operator()(int) const { return true; }
};

// intersect_point (utils/utils.py:69-151), sequential early-exit scan by one thread; `maybe(i)` as
// in intersect_point_warp below (false only for a segment the reference cannot accept)
template <class P, class F = NoPrefilter>
__device__ inline Intersect64 intersect_point64(const P& pts, int n, double qx, double qy,
                                                double r, double t, bool wrap, const F& maybe = F()) {
    Intersect64 o;
    o.px = 0.0; o.py = 0.0; o.t = 0.0; o.i = 0; o.found = 0;
    const int start_i = (int)t;                 // :78
    const double start_t = t - (double)start_i;  // == t % 1.0 for t >= 0, exactly        // :79
    double t1, t2, vx, vy;
    for (int i = start_i; i < n - 1; ++i) {     // :84
        if (!maybe(i)) continue;
        const double2 s = pts(i);
        if (!intersect_segment64(qx, qy, r, s, pts(i + 1), t1, t2, vx, vy)) continue;
        double tt = -1.0;
        if (i == start_i) {                     // :102-112
            if (t1 >= 0.0 && t1 <= 1.0 && t1 >= start_t) tt = t1;
            else if (t2 >= 0.0 && t2 <= 1.0 && t2 >= start_t) tt = t2;
        } else if (t1 >= 0.0 && t1 <= 1.0) tt = t1;   // :113
        else if (t2 >= 0.0 && t2 <= 1.0) tt = t2;     // :118
        if (tt >= 0.0) {
            o.t = tt; o.i = i; o.found = 1;
            o.px = xadd(s.x, xmul(tt, vx)); o.py = xadd(s.y, xmul(tt, vy));
            return o;
        }
    }
    if (wrap) {                                 // :124
        for (int i = -1; i < start_i; ++i) {    // :125
            if (!maybe(i)) continue;
            const double2 s = pts(pymod(i, n));
            if (!intersect_segment64(qx, qy, r, s, pts(pymod(i + 1, n)), t1, t2, vx, vy)) continue;
            double tt = -1.0;
            if (t1 >= 0.0 && t1 <= 1.0) tt = t1;        // :140
            else if (t2 >= 0.0 && t2 <= 1.0) tt = t2;   // :145
            if (tt >= 0.0) {
                o.t = tt; o.i = i; o.found = 1;
                o.px = xadd(s.x, xmul(tt, vx)); o.py = xadd(s.y, xmul(tt, vy));
                return o;
            }
        }
    }
    return o;
}

// Warp-parallel intersect_point with the same result as the sequential scan: 32 consecutive
// segments per step in the reference's scan order (forward from int(t), then the wrap loop from
// the closing segment -1), the reference's acceptance rules evaluated per lane in float64, the
// lowest accepting lane wins (== first hit of the sequential loop).  `maybe(i)` is a cheap
// conservative prefilter (false only if segment i cannot reach the circle).  Call with the whole
// warp converged; every lane returns the same result.
// `skip`: the first `skip` segments of the forward scan are known not to hit (a caller that has
// already tested them) and are not visited again.
template <class P, class F>
__device__ inline Intersect64 intersect_point_warp(const P& pts, int n, double qx, double qy,
                                                   double r, double t, bool wrap, int lane,
                                                   const F& maybe, int skip = 0) {
    Intersect64 o;
    o.px = 0.0; o.py = 0.0; o.t = 0.0; o.i = 0; o.found = 0;
    const int start_i = (int)t;                 // :78
    const double start_t = t - (double)start_i;  // == t % 1.0 for t >= 0, exactly        // :79
    for (int phase = 0; phase < (wrap ? 2 : 1); ++phase) {
        const int lo = phase == 0 ? start_i : -1;          // :84 / :125
        const int hi = phase == 0 ? n - 1 : start_i;       // exclusive
        for (int base = lo + (phase == 0 ? skip : 0); base < hi; base += 32) {
            const int i = base + lane;
            double tt = -1.0, vx = 0.0, vy = 0.0;
            double2 s = make_double2(0.0, 0.0);
            if (i < hi && maybe(i)) {
                double t1, t2;
                s = pts(pymod(i, n));
                if (intersect_segment64(qx, qy, r, s, pts(pymod(i + 1, n)), t1, t2, vx, vy)) {
                    if (phase == 0 && i == start_i) {       // :102-112
                        if (t1 >= 0.0 && t1 <= 1.0 && t1 >= start_t) tt = t1;
                        else if (t2 >= 0.0 && t2 <= 1.0 && t2 >= start_t) tt = t2;
                    } else if (t1 >= 0.0 && t1 <= 1.0) tt = t1;   // :113 / :140
                    else if (t2 >= 0.0 && t2 <= 1.0) tt = t2;     // :118 / :145
                }
            }
            const unsigned m = __ballot_sync(F1L_FULL, tt >= 0.0);
            if (m) {
                const int src = __ffs(m) - 1;
                const double px = xadd(s.x, xmul(tt, vx)), py = xadd(s.y, xmul(tt, vy));
                o.found = 1;
                o.i = base + src;
                o.t = __shfl_sync(F1L_FULL, tt, src);
                o.px = __shfl_sync(F1L_FULL, px, src);
                o.py = __shfl_sync(F1L_FULL, py, src);
                return o;
            }
        }
    }
    return o;
}

// intersect_point for a circle that is known to stay clear of every open segment (the nearest
// distance to the raceline exceeds the radius): the only segment the reference's scan can still
// accept is the closing one, i = -1 of the wrap loop (utils.py:125-150), from the last waypoint to
// the first.  One float64 segment test instead of a scan of the whole track.
template <class P>
__device__ inline Intersect64 intersect_closing_only(const P& pts, int n, double qx, double qy,
                                                     double r, bool wrap) {
    Intersect64 o;
    o.px = 0.0; o.py = 0.0; o.t = 0.0; o.i = 0; o.found = 0;
    if (!wrap) return o;
    double t1, t2, vx, vy;
    const double2 s = pts(n - 1);
    if (!intersect_segment64(qx, qy, r, s, pts(0), t1, t2, vx, vy)) return o;
    double tt = -1.0;
    if (t1 >= 0.0 && t1 <= 1.0) tt = t1;        // :140
    else if (t2 >= 0.0 && t2 <= 1.0) tt = t2;   // :145
    if (tt >= 0.0) {
        o.t = tt; o.i = -1; o.found = 1;
        o.px = xadd(s.x, xmul(tt, vx)); o.py = xadd(s.y, xmul(tt, vy));
    }
    return o;
}

// The same for one query per G-lane group (G = 8: four queries per warp) that share the point and
// the start parameter and differ in the radius -- the lookahead rows of the goal grid, whose hits
// lie a few segments ahead, so G consecutive segments per step are plenty.  Every group steps
// through the same segment sequence; a group that has its hit keeps it and idles.  `active`: the
// group has a query.  Only the first `max_steps` x G segments of the forward scan are visited:
// `pending` returns whether this group's query is still open (the caller finishes it with
// intersect_point_warp; a circle that misses the raceline scans the whole track, which 32 lanes
// do four times faster than 8).  Call with the whole warp converged; the lanes of a group return
// its result.
template <int G, class P, class F>
__device__ inline Intersect64 intersect_point_group(const P& pts, int n, double qx, double qy,
                                                    double r, double t, bool wrap, int lane,
                                                    const F& maybe, bool active, int max_steps,
                                                    bool& pending) {
    Intersect64 o;
    o.px = 0.0; o.py = 0.0; o.t = 0.0; o.i = 0; o.found = 0;
    const int gl = lane & (G - 1), gbase = lane & ~(G - 1);
    const unsigned gmask = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);
    const int start_i = (int)t;                 // :78
    const double start_t = t - (double)start_i;  // == t % 1.0 for t >= 0, exactly        // :79
    bool done = !active;
    pending = false;
    int steps = 0;
    for (int phase = 0; phase < (wrap ? 2 : 1); ++phase) {
        const int lo = phase == 0 ? start_i : -1;          // :84 / :125
        const int hi = phase == 0 ? n - 1 : start_i;       // exclusive
        for (int base = lo; base < hi; base += G) {
            if (__all_sync(F1L_FULL, done)) return o;
            if (steps++ >= max_steps) { pending = !done; return o; }
            const int i = base + gl;
            double tt = -1.0, vx = 0.0, vy = 0.0;
            double2 s = make_double2(0.0, 0.0);
            if (!done && i < hi && maybe(i)) {
                double t1, t2;
                s = pts(pymod(i, n));
                if (intersect_segment64(qx, qy, r, s, pts(pymod(i + 1, n)), t1, t2, vx, vy)) {
                    if (phase == 0 && i == start_i) {       // :102-112
                        if (t1 >= 0.0 && t1 <= 1.0 && t1 >= start_t) tt = t1;
                        else if (t2 >= 0.0 && t2 <= 1.0 && t2 >= start_t) tt = t2;
                    } else if (t1 >= 0.0 && t1 <= 1.0) tt = t1;   // :113 / :140
                    else if (t2 >= 0.0 && t2 <= 1.0) tt = t2;     // :118 / :145
                }
            }
            const unsigned m = (__ballot_sync(F1L_FULL, tt >= 0.0) >> gbase) & gmask;
            const int src = gbase + (m ? __ffs(m) - 1 : 0);
            const double px = xadd(s.x, xmul(tt, vx)), py = xadd(s.y, xmul(tt, vy));
            const double ht = __shfl_sync(F1L_FULL, tt, src);
            const double hx = __shfl_sync(F1L_FULL, px, src);
            const double hy = __shfl_sync(F1L_FULL, py, src);
            if (!done && m) {
                o.found = 1;
                o.i = base + (src - gbase);
                o.t = ht; o.px = hx; o.py = hy;
                done = true;
            }
        }
    }
    return o;
}

// get_actuation (utils/utils.py:153-161): returns steer, passes speed through
__device__ __forceinline__ double actuation_steer64(double pose_theta, double lx, double ly,
                                                    double qx, double qy, double L, double wb) {
    double sn, cs;
    sincos(-pose_theta, &sn, &cs);   // (one argument reduction; the values are those of sin() and cos())
    const double wy = xadd(xmul(sn, xsub(lx, qx)), xmul(cs, xsub(ly, qy)));
    if (fabs(wy) < 1e-6) return 0.0;                                   // :157
    const double radius = __ddiv_rn(1.0, __ddiv_rn(xmul(2.0, wy), xmul(L, L)));  // :159
    return atan(__ddiv_rn(wb, radius));                                // :160
}

// ---------------------------------------------------------------------------------------------
// packed FP32x2 helpers (sm_100 FFMA2 / FMUL2).  Values live in 64-bit registers so that ptxas
// keeps each pair in an aligned register pair across the loop (float2 halves are independent
// 32-bit values to the allocator and get MOVed together before every use).
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 fmul2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// three-input min (sm_100 FMNMX3, one ALU-pipe instruction)
__device__ __forceinline__ float fmin3(float a, float b, float c) {
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// ---------------------------------------------------------------------------------------------
// shared memory through explicit 32-bit shared-space addresses.  Under register pressure nvcc
// re-derives the address of every shared access from scratch (S2R SR_CgaCtaId + MOV + IADD3 + LEA
// for the window base, S2R SR_TID.X + shifts for the lane part: ~250 of eval_kernel's ~1400
// warp-instructions per candidate outside its hot loop, 4 of 135 inside it).  An address that went
// through `opaque()` cannot be rematerialised: it stays in its register (or is spilled and comes
// back with one LDL).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void opaque(uint32_t& v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ void opaque(int& v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ f32x2 lds64(uint32_t a) {
    f32x2 v;
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t a, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---------------------------------------------------------------------------------------------
// warp helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(F1L_FULL, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(F1L_FULL, v, o));
    return v;
}

// order-preserving float -> uint32 map (for the packed 64-bit atomicMin argmin)
__device__ __forceinline__ uint32_t float_orderable(float f) {
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float orderable_float(uint32_t u) {
    const uint32_t b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
    return __uint_as_float(b);
}
