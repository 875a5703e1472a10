// f1l_rollout.cuh -- K6: one closed-loop step of a fleet of cars (f1l_rollout_dev, f1l_rollout_st_dev).
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
//
// Two instances, one per vehicle model: Kinematic (the rear-axle kinematic bicycle) and SingleTrack
// (f1tenth_gym's dynamic single-track model, one RK4 step per substep, include/f1l.h).  They differ
// only in the motion of a live car within a substep; everything else is the same code.
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
    // single-track model only (appended: the kinematic instance reads none of it)
    double* dyn;             // [S,3] delta, yaw rate, slip angle
    double* tr_dyn;          // [S,3] dyn at the start of the step, nullable
    f1l_vehicle veh;
    // prediction (f1l_rollout_predict_dev, nullable): the next step's opponent velocities
    // [S,F1L_MAX_OPP,2], map frame, in the order of `opp`
    double* opp_vel;
};

struct Kinematic { static constexpr bool single_track = false; };
struct SingleTrack { static constexpr bool single_track = true; };

// d/dt of q = (x, y, delta, v, psi, yaw rate, beta) with (sv, acc) held; tests/st_model.py restates
// it operation for operation.  cf / cr / A1 / A2 / A3 / B1 depend on acc only (once per substep).
struct StSubstep {
    double sv, acc, cf, A1, A2, A3, B1;
};

__device__ __forceinline__ void st_deriv(const RolloutArgs& a, double L, double kr, double kb,
                                         const StSubstep& u, const double q[7], double f[7]) {
    const double d = q[2], v = q[3], psi = q[4], r = q[5], b = q[6];
    f[2] = u.sv;
    f[3] = u.acc;
    if (fabs(v) < a.veh.v_kin) {
        // kinematic form
        double sd, cd;
        sincos(d, &sd, &cd);
        const double td = __ddiv_rn(sd, cd);
        double sp, cp;
        sincos(psi, &sp, &cp);
        f[0] = fm(v, cp);
        f[1] = fm(v, sp);
        f[4] = fm(__ddiv_rn(v, L), td);
        f[5] = fa(fm(__ddiv_rn(u.acc, L), td), fm(__ddiv_rn(v, fm(fm(L, cd), cd)), u.sv));
        f[6] = 0.0;
    } else {
        double sp, cp;
        sincos(fa(psi, b), &sp, &cp);
        const double iv = __ddiv_rn(1.0, v);
        f[0] = fm(v, cp);
        f[1] = fm(v, sp);
        f[4] = r;
        f[5] = fm(kr, fs(fa(fm(u.A2, b), fm(u.A3, d)), fm(fm(u.A1, iv), r)));
        f[6] = fs(fm(fs(fm(fm(fm(kb, u.A2), iv), iv), 1.0), r), fm(fm(kb, iv), fs(fm(u.B1, b), fm(u.cf, d))));
    }
}

// one substep of a live single-track car: command -> (sv, acc), then one classical RK4 step
__device__ __forceinline__ void st_substep(const RolloutArgs& a, double steer, double target, double& x,
                                           double& y, double& th, double& v, double& dl, double& r,
                                           double& b) {
    const f1l_vehicle& p = a.veh;
    const double g = 9.81;
    const double L = fa(p.lf, p.lr);
    const double kr = __ddiv_rn(fm(p.mu, p.m), fm(p.I, L));
    const double kb = __ddiv_rn(p.mu, L);
    const double dt = a.dt;
    StSubstep u;
    u.sv = fmin(fmax(__ddiv_rn(fs(steer, dl), dt), -p.max_steer_vel), p.max_steer_vel);
    const double a_pos = v > p.v_switch ? __ddiv_rn(fm(a.max_accel, p.v_switch), v) : a.max_accel;
    u.acc = fmin(fmax(__ddiv_rn(fs(target, v), dt), -a.max_accel), a_pos);
    const double Ff = fs(fm(g, p.lr), fm(u.acc, p.h)), Fr = fa(fm(g, p.lf), fm(u.acc, p.h));
    u.cf = fm(p.C_Sf, Ff);
    const double cr = fm(p.C_Sr, Fr);
    u.A1 = fa(fm(fm(p.lf, p.lf), u.cf), fm(fm(p.lr, p.lr), cr));
    u.A2 = fs(fm(p.lr, cr), fm(p.lf, u.cf));
    u.A3 = fm(p.lf, u.cf);
    u.B1 = fa(cr, u.cf);
    const double q0[7] = {x, y, dl, v, th, r, b};
    const double hdt = fm(0.5, dt), dt6 = __ddiv_rn(dt, 6.0);
    double k[7], q[7], sum[7];
    st_deriv(a, L, kr, kb, u, q0, k);
#pragma unroll
    for (int i = 0; i < 7; ++i) { sum[i] = k[i]; q[i] = fa(q0[i], fm(hdt, k[i])); }
    st_deriv(a, L, kr, kb, u, q, k);
#pragma unroll
    for (int i = 0; i < 7; ++i) { sum[i] = fa(sum[i], fm(2.0, k[i])); q[i] = fa(q0[i], fm(hdt, k[i])); }
    st_deriv(a, L, kr, kb, u, q, k);
#pragma unroll
    for (int i = 0; i < 7; ++i) { sum[i] = fa(sum[i], fm(2.0, k[i])); q[i] = fa(q0[i], fm(dt, k[i])); }
    st_deriv(a, L, kr, kb, u, q, k);
#pragma unroll
    for (int i = 0; i < 7; ++i) sum[i] = fa(sum[i], k[i]);
    x = fa(q0[0], fm(dt6, sum[0]));
    y = fa(q0[1], fm(dt6, sum[1]));
    dl = fa(q0[2], fm(dt6, sum[2]));
    v = fa(q0[3], fm(dt6, sum[3]));
    th = fa(q0[4], fm(dt6, sum[4]));
    r = fa(q0[5], fm(dt6, sum[5]));
    b = fa(q0[6], fm(dt6, sum[6]));
}

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

template <class Model>
__global__ void __launch_bounds__(ROLLOUT_WARPS * 32) rollout_step_kernel(RolloutArgs a) {
    constexpr bool ST = Model::single_track;
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
    unsigned st_end = 0;   // prediction: the car's status and slip angle after this pass
    double beta = 0.0;

    if (!a.steer_speed) {
        if (a.opp_vel) {
            st_end = a.status[car];
            if constexpr (ST) beta = a.dyn[3 * (size_t)car + 2];
        }
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
        double dl = 0.0, r = 0.0, b = 0.0;   // single-track: delta, yaw rate, slip angle
        if constexpr (ST) {
            dl = a.dyn[3 * (size_t)car];
            r = a.dyn[3 * (size_t)car + 1];
            b = a.dyn[3 * (size_t)car + 2];
        }
        if (live) {
            if constexpr (ST) {
                if (a.tr_dyn) {
                    double* o = a.tr_dyn + 3 * (size_t)car;
                    o[0] = dl; o[1] = r; o[2] = b;
                }
            }
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
                v = 0.0;   // frozen: keeps its pose (and steering angle)
                if constexpr (ST) { r = 0.0; b = 0.0; }
            } else if constexpr (ST) {
                st_substep(a, steer, target, x, y, th, v, dl, r, b);
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
            if (st & (F1L_CAR_HIT_MAP | F1L_CAR_HIT_CAR)) {
                v = 0.0;
                if constexpr (ST) { r = 0.0; b = 0.0; }
            }
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
            if constexpr (ST) {
                double* d = a.dyn + 3 * (size_t)car;
                d[0] = dl; d[1] = r; d[2] = b;
            }
            a.status[car] = (uint8_t)st;
            a.progress[car] = prog;
            a.track_i[car] = ti;
            a.track_s[car] = ts;
            if (a.tr_status) a.tr_status[car] = (uint8_t)st;
            if (a.tr_progress) a.tr_progress[car] = prog;
        }
        st_end = st;
        beta = b;
    }
    // the car's velocity as its opponents predict it: along the heading (kinematic) or the course
    // psi + beta (single-track); a frozen car stands
    double vx = 0.0, vy = 0.0;
    if (a.opp_vel && !(st_end & (F1L_CAR_HIT_MAP | F1L_CAR_HIT_CAR))) {
        double sc, cc;
        sincos(ST ? fa(th, beta) : th, &sc, &cc);
        vx = fm(v, cc);
        vy = fm(v, sc);
    }
    // the next step's opponents of this car: the other cars of its race in race order
    int k = 0;
    for (int j = 0; j < G; ++j) {   // uniform
        const double xj = __shfl_sync(F1L_FULL, x, j), yj = __shfl_sync(F1L_FULL, y, j);
        const double tj = __shfl_sync(F1L_FULL, th, j);
        const double vxj = __shfl_sync(F1L_FULL, vx, j), vyj = __shfl_sync(F1L_FULL, vy, j);
        if (live && j != lane) {
            double* o = a.opp + 3 * ((size_t)car * F1L_MAX_OPP + k);
            o[0] = xj; o[1] = yj; o[2] = tj;
            if (a.opp_vel) {
                double* ov = a.opp_vel + 2 * ((size_t)car * F1L_MAX_OPP + k);
                ov[0] = vxj; ov[1] = vyj;
            }
            ++k;
        }
    }
    if (live) a.n_opp[car] = G - 1;
}
