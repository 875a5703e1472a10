// f1l_rollout.cuh -- K6: one closed-loop step of a fleet of kinematic-bicycle cars (f1l_rollout_dev).
//
// After the batch pipeline (sampler -> eval -> select) has planned every car of the fleet, this
// kernel turns each car's (steer, speed) command into motion, tests the new poses against the map
// and the other cars of its race, tracks raceline progress and writes the opponent table the next
// step's sampler reads.  Replaces the user loop around the planner (lattice_planner.py:204-214 and
// the gym step of examples/control/pure_pursuit.py:47-57).
//
// One warp per race of G <= 17 consecutive cars, one lane per car.  All lanes of a race go through
// the substeps together, so the car-to-car tests and the opponent table take the other cars' poses
// from __shfl_sync: no global-memory exchange between cars.
#pragma once
#include "f1l_common.cuh"
#include "f1l_lattice.cuh"

#define ROLLOUT_WARPS 4   // races per CTA

struct RolloutArgs {
    TrackView tr;
    GridView grid;
    const double2* seg_s;   // [n-1] (cumulative length at the segment's start, segment length)
    double lap;             // cumulative length of the n-1 segments + the closing gap p_{n-1} -> p_0
    double res;             // grid resolution (cell = floor((p - origin) / res))
    int has_grid, collision_mode;
    double hl, hw, disc_off, wheelbase;   // half footprint, disc spacing L/3
    double dt, max_steer, max_accel, v_max;
    int substeps, group, n_races;
    // fleet (in / out)
    double* state;          // [S,4] x, y, theta, v
    uint8_t* status;        // [S] F1L_CAR_*
    double* progress;       // [S]
    int32_t* track_i;       // [S] tracked raceline segment (< 0: re-acquire from near_i / near4)
    double* track_s;        // [S] arc length at the tracked point
    // this step's plan (null: the initial pass of a call, no integration)
    const double* steer_speed;   // [S,2]
    const float* best_cost;      // [S]
    // initial pass: global nearest_point of every car (K1)
    const int32_t* near_i;       // [S]
    const double* near4;         // [S,4] proj_x, proj_y, dist, t
    // opponent table of the next step: [S,F1L_MAX_OPP,3] map-frame (x, y, theta), [S] count
    double* opp;
    int32_t* n_opp;
    // trace rows of this step, each nullable
    double* tr_state;        // [S,4] state at the start of the step
    double* tr_ss;           // [S,2] raw command
    uint8_t* tr_status;      // [S] after the step
    double* tr_progress;     // [S] after the step
};

// the footprint's map predicate of collision_mode, in float64 in the map frame
__device__ __forceinline__ bool rollout_map_hit(const RolloutArgs& a, double x, double y, double c,
                                                double s) {
    const GridView& g = a.grid;
    if (a.collision_mode == 1) {
        // three discs: centre and +-L/3 along the body axis, one distance-transform lookup each
        const double lx = fm(a.disc_off, c), ly = fm(a.disc_off, s);
        bool hit = false;
#pragma unroll
        for (int k = -1; k <= 1; ++k) {
            const double px = fa(x, fm((double)k, lx)), py = fa(y, fm((double)k, ly));
            const int col = floor_int(__ddiv_rn(fs(px, g.ox), a.res));
            const int row = floor_int(__ddiv_rn(fs(py, g.oy), a.res));
            if ((unsigned)col >= (unsigned)g.w || (unsigned)row >= (unsigned)g.h) hit = true;
            else if ((int)__ldg(g.edt2 + (size_t)row * g.w + col) < g.disc_t2) hit = true;
        }
        return hit;
    }
    // nine probes: corners, edge mid-points and centre, centre + sa * l-axis + sb * w-axis
    const double lx = fm(a.hl, c), ly = fm(a.hl, s);
    const double wx = -fm(a.hw, s), wy = fm(a.hw, c);
    bool hit = false;
#pragma unroll
    for (int p = 0; p < 9; ++p) {
        const double sa = (double)(p / 3 - 1), sb = (double)(p % 3 - 1);
        const double px = fa(fa(x, fm(sa, lx)), fm(sb, wx));
        const double py = fa(fa(y, fm(sa, ly)), fm(sb, wy));
        hit |= grid_hit(g.occ, g.w, g.h, 0, 0, __ddiv_rn(fs(px, g.ox), a.res), __ddiv_rn(fs(py, g.oy), a.res));
    }
    return hit;
}

__global__ void __launch_bounds__(ROLLOUT_WARPS * 32) rollout_step_kernel(RolloutArgs a) {
    const int lane = threadIdx.x & 31;
    const int race = blockIdx.x * ROLLOUT_WARPS + (threadIdx.x >> 5);
    if (race >= a.n_races) return;   // warp-uniform
    const int G = a.group;
    const bool live = lane < G;
    const int car = race * G + (live ? lane : 0);
    double x = a.state[4 * (size_t)car], y = a.state[4 * (size_t)car + 1];
    double th = a.state[4 * (size_t)car + 2], v = a.state[4 * (size_t)car + 3];
    int ti = a.track_i[car];
    double ts = a.track_s[car];

    if (!a.steer_speed) {
        // initial pass of a call: re-acquire lost cars on the whole raceline
        if (ti < 0) {
            ti = a.near_i[car];
            const double2 ss = a.seg_s[ti];
            ts = fa(ss.x, fm(a.near4[4 * (size_t)car + 3], ss.y));
            if (live) { a.track_i[car] = ti; a.track_s[car] = ts; }
        }
    } else {
        unsigned st = a.status[car] & ~F1L_CAR_NO_FEASIBLE;
        const double cmd_steer = a.steer_speed[2 * (size_t)car], cmd_speed = a.steer_speed[2 * (size_t)car + 1];
        const double steer = fmin(fmax(cmd_steer, -a.max_steer), a.max_steer);
        double target = 0.0;
        if (a.best_cost[car] < CUDART_INF_F) target = fmin(cmd_speed, a.v_max);
        else st |= F1L_CAR_NO_FEASIBLE;
        if (live) {
            if (a.tr_state) {
                double2* o = reinterpret_cast<double2*>(a.tr_state + 4 * (size_t)car);
                o[0] = make_double2(x, y);
                o[1] = make_double2(th, v);
            }
            if (a.tr_ss) *reinterpret_cast<double2*>(a.tr_ss + 2 * (size_t)car) = make_double2(cmd_steer, cmd_speed);
        }
        const double dv = fm(a.max_accel, a.dt);
        const double yaw = tan(steer);   // once per step
        const double c_hl = a.hl, c_hw = a.hw;
        for (int k = 0; k < a.substeps; ++k) {
            if (st & (F1L_CAR_HIT_MAP | F1L_CAR_HIT_CAR)) {
                v = 0.0;   // frozen: keeps its pose
            } else {
                v = fa(v, fmin(fmax(fs(target, v), -dv), dv));
                x = fa(x, fm(fm(v, cos(th)), a.dt));
                y = fa(y, fm(fm(v, sin(th)), a.dt));
                th = fa(th, fm(fm(__ddiv_rn(v, a.wheelbase), yaw), a.dt));
            }
            double c, s;
            sincos(th, &s, &c);
            if (a.has_grid && rollout_map_hit(a, x, y, c, s)) st |= F1L_CAR_HIT_MAP;
            // the other cars of the race at their new poses (touching = free)
            for (int j = 0; j < G; ++j) {   // uniform
                const double xj = __shfl_sync(F1L_FULL, x, j), yj = __shfl_sync(F1L_FULL, y, j);
                const double cj = __shfl_sync(F1L_FULL, c, j), sj = __shfl_sync(F1L_FULL, s, j);
                if (j != lane && sat_collide(fs(xj, x), fs(yj, y), c, s, cj, sj, c_hl, c_hw)) st |= F1L_CAR_HIT_CAR;
            }
            if (st & (F1L_CAR_HIT_MAP | F1L_CAR_HIT_CAR)) v = 0.0;
        }
        // raceline progress: nearest segment in a 32-segment window starting 4 behind the tracked
        // one, cyclic over the n-1 segments, first minimum in window order (nearest_point's own
        // float64 operations); the arc-length increment is wrapped into [-lap/2, lap/2)
        const int nseg = a.tr.n - 1;
        const int nw = min(32, nseg);
        int j = (ti - 4) % nseg;
        if (j < 0) j += nseg;
        double bd = CUDART_INF, bt = 0.0;
        int bi = j;
        for (int w = 0; w < nw; ++w) {
            const double2 p0 = a.tr.xy[j], p1 = a.tr.xy[j + 1];
            double px, py, d, t;
            nearest_segment64(x, y, p0.x, p0.y, p1.x, p1.y, px, py, d, t);
            if (d < bd) { bd = d; bi = j; bt = t; }
            if (++j == nseg) j = 0;
        }
        const double2 ss = a.seg_s[bi];
        const double s_new = fa(ss.x, fm(bt, ss.y));
        double ds = fs(s_new, ts);
        if (ds >= 0.5 * a.lap) ds = fs(ds, a.lap);
        else if (ds < -0.5 * a.lap) ds = fa(ds, a.lap);
        ti = bi;
        ts = s_new;
        if (live) {
            const double prog = fa(a.progress[car], ds);
            double2* o = reinterpret_cast<double2*>(a.state + 4 * (size_t)car);
            o[0] = make_double2(x, y);
            o[1] = make_double2(th, v);
            a.status[car] = (uint8_t)st;
            a.progress[car] = prog;
            a.track_i[car] = ti;
            a.track_s[car] = ts;
            if (a.tr_status) a.tr_status[car] = (uint8_t)st;
            if (a.tr_progress) a.tr_progress[car] = prog;
        }
    }
    // the next step's opponents of this car: the other cars of its race in race order
    int k = 0;
    for (int j = 0; j < G; ++j) {   // uniform
        const double xj = __shfl_sync(F1L_FULL, x, j), yj = __shfl_sync(F1L_FULL, y, j);
        const double tj = __shfl_sync(F1L_FULL, th, j);
        if (live && j != lane) {
            double* o = a.opp + 3 * ((size_t)car * F1L_MAX_OPP + k);
            o[0] = xj; o[1] = yj; o[2] = tj;
            ++k;
        }
    }
    if (live) a.n_opp[car] = G - 1;
}
