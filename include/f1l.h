/*
 * f1l.h -- C-ABI of the B200-native lattice-planner hot path.
 *
 * The reference (f1tenth/f1tenth_planning) has no FFI: its boundary is the
 * Python API.  Every entry point below names the reference interface it
 * replaces (paths relative to the reference checkout).  The Python package
 * f1tenth_planning_b200 binds these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 (F1L_OK) or a negative f1l_status; nothing
 *     throws across the ABI; f1l_strerror() names the code.
 *   - the caller owns every buffer it passes; the handle owns the device
 *     copies of track / grid / LUT / previous path and all scratch.
 *   - "*_dev" entry points take DEVICE pointers and enqueue on the caller's
 *     stream without synchronising; the others take HOST pointers, do their
 *     own H2D/D2H on the handle's stream and synchronise it before returning.
 *   - one handle per device; a handle is not thread-safe; handles are
 *     independent of each other.
 *   - all angles in radians, lengths in metres, arrays row-major.
 */
#ifndef F1L_H
#define F1L_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct f1l_ctx* f1l_handle;

typedef enum {
    F1L_OK = 0,
    F1L_ERR_INVALID_ARG = -1,
    F1L_ERR_NO_TRACK = -2,
    F1L_ERR_CUDA = -3,
    F1L_ERR_NO_DEVICE = -4,
    F1L_ERR_TOO_LARGE = -5,
    F1L_ERR_NO_GOALS = -6,
    F1L_ERR_ALLOC = -7,
    F1L_ERR_PEER_TIMEOUT = -8
} f1l_status;

#define F1L_N_TERMS 5       /* length, max|kappa|, mean|kappa|, similarity, raceline deviation */
#define F1L_MAX_OPP 16      /* opponents per scenario */
#define F1L_MAX_M 256       /* arc samples per candidate */

/* per-candidate flag bits (flags output) */
#define F1L_FLAG_VALID 1u        /* Newton converged, s_f > 0, finite, max|kappa| <= kappa_max */
#define F1L_FLAG_COLLIDE_OPP 2u  /* footprint overlaps an opponent rectangle */
#define F1L_FLAG_COLLIDE_MAP 4u  /* a footprint probe hits an occupied / out-of-bounds cell */
#define F1L_FLAG_NO_CENTRE 8u    /* lookahead circle found no raceline intersection for this row */
#define F1L_FLAG_PASS_SHIFT 4    /* bits 4..7: Newton quadrature passes this candidate used */

/*
 * Planner configuration.  Replaces the constructor kwargs / hard-coded numbers
 * of the reference: LatticePlanner.__init__ (planning/lattice_planner/
 * lattice_planner.py:44-55), samples per trajectory =100 (:197), tracker
 * lookahead =0.8 (:211), the undefined N_SHIFT/N_CULL/NUM_STEPS globals of the
 * cost helpers (:273-296), vehicle footprint LENGTH/WIDTH
 * (control/kinematic_mpc/kinematic_mpc.py:60-61).
 */
typedef struct {
    int32_t n_samples;       /* M, arc samples per candidate (2..F1L_MAX_M); ref 100 */
    int32_t n_newton;        /* fixed Newton iterations per candidate; default 8 */
    int32_t window;          /* W raceline-deviation window in segments; <=0 or >=N-1 -> all N-1 */
    int32_t n_shift;         /* similarity cost: shift of the previous path; default 5 */
    int32_t n_cull;          /* similarity cost: samples culled from the tail; default 10 */
    int32_t literal_tracker; /* 1: reproduce lattice_planner.py:208-212 literally (map pose vs
                                vehicle-frame trajectory, "speed" = theta column) */
    int32_t use_goal_kappa;  /* 1: end curvature p3 = raceline kappa at the goal centre; 0: p3 = 0 */
    int32_t generator;       /* 0: cubic spiral (LUT seed + Newton on p1, p2, s_f); 1: G1 clothoid as
                                the reference's Clothoid.G1Hermite(0,0,0,gx,gy,gtheta)
                                (lattice_planner.py:196), 1-D Newton */
    int32_t prune_window;    /* raceline deviation: 0 = every sample against every window segment
                                (default); 1 = skip the window segments that provably cannot be
                                nearest to any sample of the candidate (chord-midpoint bound).
                                Same minima, hence bit-identical costs, fewer segment tests.
                                A candidate that collided (cost +inf) skips the deviation pass
                                altogether unless the per-term costs were requested. */
    int32_t collision_mode;  /* occupancy-grid collision test of a footprint (map_collision stub,
                                utils/utils.py:297-301): 0 = nine probe points (corners, edge
                                mid-points, centre; default); 1 = three discs along the body axis
                                (centres -L/3, 0, +L/3, radius sqrt((L/6)^2 + (W/2)^2): they cover
                                the rectangle), ONE lookup each in a Euclidean distance transform of
                                the grid built at f1l_set_grid -- a disc collides iff the distance
                                (in cells, between cell centres) from its centre's cell to the
                                nearest occupied / out-of-bounds cell is at most radius/res + sqrt 2
                                (half a cell diagonal for the centre within its cell, half for the
                                extent of the occupied cell): strictly conservative, every
                                nine-probe collision is a disc collision */
    double weights[F1L_N_TERMS]; /* cost weights (lattice_planner.py:130-156) */
    double kappa_max;        /* candidates with max|kappa| above it are invalid; <=0 disables */
    double car_length;       /* 0.58 */
    double car_width;        /* 0.31 */
    double converge_tol;     /* endpoint tolerance: |end - goal| < tol*max(1,|goal|); default 1e-4 */
    double tracker_lookahead;/* 0.8 (lattice_planner.py:211) */
    double wheelbase;        /* 0.33 */
    double max_reacquire;    /* 20.0 (pure_pursuit.py:52) */
} f1l_config;

/* Fills *cfg with the defaults named above. */
int f1l_default_config(f1l_config* cfg);

/* Create / destroy the per-device planner state.  Replaces LatticePlanner.__init__
 * (lattice_planner.py:44-55) and PurePursuitPlanner.__init__ (pure_pursuit.py:51-54).
 * Builds the cubic-spiral seed LUT on the device (see f1l_get_lut).  Single queries write their
 * results straight into a mapped pinned host block: if the device cannot map it
 * (cudaHostGetDevicePointer fails), f1l_create returns F1L_ERR_CUDA and creates no handle. */
int f1l_create(f1l_handle* out, int device, const f1l_config* cfg);
int f1l_destroy(f1l_handle h);
const char* f1l_strerror(int code);
int f1l_set_config(f1l_handle h, const f1l_config* cfg);
int f1l_get_config(f1l_handle h, f1l_config* cfg);
int f1l_device(f1l_handle h);
/* Last CUDA error string seen by this handle ("" if none). */
const char* f1l_last_cuda_error(f1l_handle h);

/* Track upload.  wpts is [N, ncols] float64 row-major, columns x, y[, v, psi, kappa]
 * (examples/control/Spielberg_raceline.csv:1; pure_pursuit.py:101 uses col 2 as speed).
 * Replaces `self.waypoints = waypoints` (lattice_planner.py:49, pure_pursuit.py:54,103).
 * Slow path: besides the device copies, a track of up to 2560 segments is also written into the
 * device's constant-memory line-form table that the batched nearest_point scan prefers (one table
 * per device, owned by the handle that uploaded last; other handles on the device scan their
 * global-memory copy, same results).  The call synchronises the whole device first. */
int f1l_set_track(f1l_handle h, const double* wpts, int n, int ncols);

/* Occupancy grid upload: occ is [H, W] uint8 row-major, 0 = free, non-zero = occupied,
 * cell (row, col) covers [ox+col*res, ox+(col+1)*res) x [oy+row*res, ...).
 * Replaces the map_collision stub (utils/utils.py:297-301). */
int f1l_set_grid(f1l_handle h, const uint8_t* occ, int height, int width,
                 double origin_x, double origin_y, double resolution);
int f1l_clear_grid(f1l_handle h);
/* The Euclidean distance transform collision_mode = 1 looks up: out [H, W] uint16 = squared
 * distance in cells from each cell to the nearest occupied or out-of-bounds cell, exact up to
 * 24^2 = 576, 577 = farther.  Built on the device by f1l_set_grid. */
int f1l_get_edt(f1l_handle h, uint16_t* out);

/* Goal grid of the built-in sampler: lookahead distances x lateral widths.
 * Replaces the kwargs of sample_lookahead_square (lattice_planner.py:228-229).
 * Candidate index c = j*n_widths + k (lookahead-major). */
int f1l_set_goal_grid(f1l_handle h, const double* lookaheads, int n_lookaheads,
                      const double* widths, int n_widths);

/* Spiral seed LUT [nx, ny, nt, 4] float32 = (p1, p2, s_f, converged) over local goals
 * x in [x0,x1], y in [y0,y1], theta in [t0,t1].  The handle builds it on the device at
 * f1l_create; these read it back / replace it.  dims/ranges: int[3], double[6]. */
int f1l_get_lut_shape(f1l_handle h, int32_t dims[3], double ranges[6]);
int f1l_get_lut(f1l_handle h, float* lut_out);
int f1l_set_lut(f1l_handle h, const float* lut, const int32_t dims[3], const double ranges[6]);

/* Previous plan for the similarity cost (lattice_planner.py:287-296 `prev_path`):
 * theta column of the previous best trajectory, vehicle frame of the previous call.
 * f1l_plan stores it automatically; these override / clear it. */
int f1l_set_prev_path(f1l_handle h, const float* theta_prev, int m);
int f1l_clear_prev_path(f1l_handle h);

/*
 * Result of one planning query (host memory, filled by f1l_plan*).
 * The optional arrays may be NULL to skip that download.
 */
typedef struct {
    /* scalars */
    double steer;            /* tracker output (pure_pursuit.py:122 order: steer, speed) */
    double speed;
    int32_t best_idx;        /* argmin candidate, ties -> lowest index (lattice_planner.py:169-171) */
    int32_t no_feasible;     /* 1 if every candidate cost is +inf (best_idx = 0) */
    int32_t tracker_found;   /* 0 -> "Cannot find lookahead point" (pure_pursuit.py:112-114) */
    int32_t n_candidates;    /* C */
    float best_cost;
    int32_t reserved;
    /* arrays, caller-allocated */
    float* best_traj;        /* [M,4] x, y, theta, kappa(signed) in the vehicle frame */
    float* costs;            /* [C] total cost, +inf for invalid / collided */
    float* terms;            /* [C,5] per-term costs (unweighted) */
    uint8_t* flags;          /* [C] F1L_FLAG_* */
    float* goals;            /* [C,3] local goals (x, y, theta) fed to the generator */
    float* params;           /* [C,4] solved spiral (p1, p2, s_f, p3) */
    float* states;           /* [C,M,4] every trajectory (debug / custom cost functions) */
    float* headings;         /* [C,M,2] (cos, sin) of the sample headings used by the footprint
                                (teacher-forced collision tests) */
    double* best_traj_map;   /* [M,4] the best trajectory in the MAP frame with a speed column,
                                (X, Y, v, Theta): X = pose + R(theta_pose) (x, y), Theta = theta +
                                theta_pose, v = raceline speed at the goal centre (explicit goals:
                                the ego speed).  The form a map-frame tracker consumes -- the
                                reference hands its tracker the vehicle-frame array against a
                                map-frame pose (lattice_planner.py:208-212, SURVEY A.7 / B.8). */
} f1l_plan_result;

/*
 * One planning query: sampler -> spiral generation -> fused cost + collision -> argmin ->
 * tracker.  Replaces LatticePlanner.plan (lattice_planner.py:174-214).
 * pose = (x, y, theta, velocity) map frame; opp = [K,3] map-frame (x, y, theta) or NULL.
 * update_prev != 0 stores the best trajectory's theta column as the next call's prev_path.
 */
int f1l_plan(f1l_handle h, const double pose[4], const double* opp, int n_opp,
             int update_prev, f1l_plan_result* out);

/*
 * f1l_plan against MOVING opponents: opponent k, at opp[k] = (x, y, theta) now, moves at the
 * constant map-frame velocity opp_vel[k] = (vx, vy) m/s and keeps its heading: its centre at time
 * t is (x + vx t, y + vy t).  The ego is timed along each candidate at v_e = max(pose[3], v_min):
 * sample i of M on a candidate of length s_f is reached at t_i = i s_f / ((M - 1) v_e), and every
 * sample's footprint is tested against the opponents' footprints at t_i.  In float32 as the
 * kernel computes it: k_t = (float)(1 / ((M - 1) v_e)) and the velocities rotated into the vehicle
 * frame (wx, wy) in float64, then per candidate dt = s_f * k_t and per sample t_i = (float)i * dt,
 * centre (ox + wx t_i, oy + wy t_i), each operation rounded on its own.  With every velocity zero
 * the result is bit-identical to f1l_plan.  v_min must be finite and > 0 (a car at rest would
 * otherwise never arrive anywhere); opp_vel [n_opp,2] f64 may be NULL only when n_opp = 0, and
 * every velocity must be finite (a NaN would clear a collision): else F1L_ERR_INVALID_ARG.
 */
int f1l_plan_motion(f1l_handle h, const double pose[4], const double* opp, const double* opp_vel,
                    int n_opp, double v_min, int update_prev, f1l_plan_result* out);

/* Same, but only candidates [c_begin, c_end) are evaluated (candidate sharding of one dense
 * query across GPUs; best_idx is still the global index).  Without attached peers the result is
 * the winner of the shard; with f1l_xchg_attach it is the winner over all ranks' shards. */
int f1l_plan_shard(f1l_handle h, const double pose[4], const double* opp, int n_opp,
                   int c_begin, int c_end, f1l_plan_result* out);

/* Row-interleaved shard: only the lookahead rows row_begin, row_begin + row_step, ... of the goal
 * grid are evaluated (all widths of each).  Near and far goals cost differently (short spirals
 * fail validation early, long ones meet more opponents and walls), so rank r of W taking rows
 * r, r + W, ... balances the ranks where contiguous blocks do not.  Indices stay global; the
 * peer exchange applies as for f1l_plan_shard.  0 <= row_begin < row_step.  A rank whose
 * row_begin is beyond the last row (more ranks than rows) evaluates nothing: with peers attached
 * it still joins the exchange and returns the global winner, alone it is F1L_ERR_INVALID_ARG.
 * update_prev != 0
 * stores the winner's theta column as the next call's prev_path like f1l_plan -- the winner of
 * this call, i.e. the global one only with peers attached (every rank then stores the same). */
int f1l_plan_rows(f1l_handle h, const double pose[4], const double* opp, int n_opp,
                  int row_begin, int row_step, int update_prev, f1l_plan_result* out);

/*
 * Peer-memory exchange for f1l_plan_shard (SURVEY 8e: "final step = gather of G (cost, idx)
 * pairs"; replaces an 8-byte NCCL all-gather plus host min).  Each rank (one PROCESS per rank --
 * CUDA IPC handles cannot be opened by the process that exported them; ranks may share a GPU)
 * exports a 3 KB block of its HBM (per-rank key + goal-centre entries, arrival counters) as a CUDA IPC handle
 * (f1l_xchg_export, 64 bytes), the caller gathers the `world` handles by any means (the Python
 * layer uses torch.distributed) and attaches them in rank order (f1l_xchg_attach: maps the peers'
 * blocks over NVLink P2P).  From then on f1l_plan_shard / f1l_plan_rows are collective: every rank calls it for
 * the same query with its own [c_begin, c_end), the select kernel pushes the rank's packed
 * (cost, index) minimum into every peer's block with system-scope atomics and waits for all
 * arrivals, and every rank returns the GLOBAL best_idx / best_cost / best_traj / steer / speed.
 * A peer that does not arrive within ~2 s yields F1L_ERR_PEER_TIMEOUT (the GPU never hangs); the
 * condition is sticky -- the ranks' call numbers no longer agree -- until every rank has detached,
 * exported and attached again.
 * All ranks must have attached before the first collective call and must stop calling before
 * any of them detaches or is destroyed (barrier on the caller's side).  world <= 16.
 */
int f1l_xchg_export(f1l_handle h, uint8_t* handle_out, int n);   /* n >= 64 */
int f1l_xchg_attach(f1l_handle h, int rank, int world, const uint8_t* handles /* [world][64] */);
int f1l_xchg_detach(f1l_handle h);

/* Same pipeline with caller-supplied local goals [C,3] (vehicle frame) instead of the built-in
 * sampler.  Replaces the user `sample_func` plug-in (lattice_planner.py:77-98,113-128). */
int f1l_plan_goals(f1l_handle h, const double pose[4], const double* goals, int n_goals,
                   const double* opp, int n_opp, int update_prev, f1l_plan_result* out);

/* Selection made by the caller (the reference's `selection_func` / `cost_funcs` plug-ins,
 * lattice_planner.py:57-75,100-111,159-172, which are user Python code): regenerates candidate
 * `idx` of the LAST f1l_plan / f1l_plan_goals query on this handle and runs the tracker on it
 * exactly as the built-in selection would (literal_tracker, wheelbase, max_reacquire, raceline
 * speed), filling steer / speed / tracker_found / best_idx / best_cost (= `cost`, no_feasible =
 * !(cost < inf)) / best_traj / best_traj_map of *out; the per-candidate arrays are not touched.
 * F1L_ERR_INVALID_ARG if no query has run since the last upload / configuration change or idx is
 * out of range. */
int f1l_select_candidate(f1l_handle h, int idx, float cost, int update_prev, f1l_plan_result* out);

/* Trajectory generation only: goals [C,3] -> states [C,M,4], params [C,4], flags [C] (host).
 * Replaces the Clothoid.G1Hermite + sample_traj loop (lattice_planner.py:195-198,
 * utils/utils.py:285-295) for user cost functions evaluated on the host. */
int f1l_generate(f1l_handle h, const double* goals, int n_goals,
                 float* states, float* params, uint8_t* flags);

/*
 * Batch of S independent scenarios, device buffers, caller's stream, no sync.
 *   poses_dev [S,4] f64, opp_dev [S,max_opp,3] f64, n_opp_dev [S] i32 (NULL -> all max_opp)
 * outputs (any may be NULL):
 *   best_idx [S] i32, best_cost [S] f32, best_traj [S,M,4] f32, costs [S,C] f32,
 *   flags [S,C] u8, steer_speed [S,2] f64
 */
int f1l_plan_batch_dev(f1l_handle h, const double* poses_dev, const double* opp_dev,
                       const int32_t* n_opp_dev, int n_scenarios, int max_opp,
                       int32_t* best_idx_dev, float* best_cost_dev, float* best_traj_dev,
                       float* costs_dev, uint8_t* flags_dev, double* steer_speed_dev,
                       void* stream);

/* Same with HOST buffers: chunked H2D -> kernels -> D2H pipeline on the handle's streams,
 * synchronised before returning. */
int f1l_plan_batch(f1l_handle h, const double* poses, const double* opp,
                   const int32_t* n_opp, int n_scenarios, int max_opp,
                   int32_t* best_idx, float* best_cost, float* best_traj,
                   float* costs, uint8_t* flags, double* steer_speed);

/*
 * Batch with a previous path per scenario: the batched form of `prev_path` of
 * get_similarity_cost (lattice_planner.py:287-296), which f1l_plan keeps on the handle for a
 * single query.  Scenario s gives bit-identically the answer of f1l_plan on this handle after
 * f1l_set_prev_path(prev_theta[s]), or after f1l_clear_prev_path when has_prev[s] == 0.
 *   prev_theta [S,M] f32 (M = n_samples, as for f1l_set_prev_path): theta column of each
 *       scenario's previous best trajectory, read; with update_prev != 0 overwritten in place with
 *       the theta column of best_traj[s] -- what f1l_plan(..., update_prev = 1) stores, also for
 *       a scenario without a feasible candidate.
 *   has_prev [S] u8 or NULL (every scenario has a path): read; with update_prev != 0 set to 1.
 * The handle's own previous path is neither read nor written.  F1L_ERR_INVALID_ARG when
 * update_prev or has_prev is given without prev_theta.  Other arguments as f1l_plan_batch_dev.
 */
int f1l_plan_batch_prev_dev(f1l_handle h, const double* poses_dev, const double* opp_dev,
                            const int32_t* n_opp_dev, int n_scenarios, int max_opp,
                            float* prev_theta_dev, uint8_t* has_prev_dev, int update_prev,
                            int32_t* best_idx_dev, float* best_cost_dev, float* best_traj_dev,
                            float* costs_dev, uint8_t* flags_dev, double* steer_speed_dev,
                            void* stream);

/* Same with HOST buffers, through the chunked pipeline of f1l_plan_batch: each chunk's paths and
 * flags travel with its other inputs and, with update_prev, come back with its other outputs.
 * Synchronised before returning. */
int f1l_plan_batch_prev(f1l_handle h, const double* poses, const double* opp,
                        const int32_t* n_opp, int n_scenarios, int max_opp,
                        float* prev_theta, uint8_t* has_prev, int update_prev,
                        int32_t* best_idx, float* best_cost, float* best_traj,
                        float* costs, uint8_t* flags, double* steer_speed);

/*
 * One batch call with every input and output in a struct: the previous paths of
 * f1l_plan_batch_prev_dev, cost weights per scenario and the per-term costs.  The four batch
 * calls above are this call with weights and terms NULL.
 *   weights [S,F1L_N_TERMS] f32 or NULL (every scenario uses the config's weights): scenario s
 *       gives bit-identically what f1l_plan gives on this handle after f1l_set_config with
 *       weights = (double) weights[s], together with the previous-path rule of
 *       f1l_plan_batch_prev_dev.  Weights are used as given, as the config's are: a non-finite
 *       weighted sum makes the candidate's cost +inf.
 *   terms [S,C,F1L_N_TERMS] f32 or NULL: the unweighted per-term costs, as f1l_plan_result.terms.
 *       With prune_window = 1, requesting them makes collided candidates scan the raceline window
 *       too (see f1l_config.prune_window).
 * F1L_ERR_INVALID_ARG for a NULL handle, call or poses, n_scenarios <= 0, max_opp outside
 * 0..F1L_MAX_OPP (or > 0 without opp), and update_prev or has_prev without prev_theta.
 * `reserved` is ignored.
 */
typedef struct {
    const double* poses;    /* [S,4] */
    const double* opp;      /* [S,max_opp,3] or NULL */
    const int32_t* n_opp;   /* [S] or NULL */
    int32_t n_scenarios, max_opp;
    float* prev_theta;      /* [S,M] or NULL, as f1l_plan_batch_prev_dev */
    uint8_t* has_prev;      /* [S] or NULL */
    int32_t update_prev, reserved;
    const float* weights;   /* [S,F1L_N_TERMS] or NULL: every scenario uses the config's weights */
    /* outputs, each nullable */
    int32_t* best_idx; float* best_cost; float* best_traj; float* costs; uint8_t* flags;
    double* steer_speed;
    float* terms;           /* [S,C,F1L_N_TERMS] unweighted per-term costs, as f1l_plan_result.terms */
} f1l_batch_call;

/* Device buffers, caller's stream, no sync (as f1l_plan_batch_dev). */
int f1l_plan_batch_call_dev(f1l_handle h, const f1l_batch_call* b, void* stream);
/* Host buffers, through the chunked pipeline of f1l_plan_batch: weights travel with each chunk's
 * inputs, terms come back with its outputs.  Synchronised before returning. */
int f1l_plan_batch_call(f1l_handle h, const f1l_batch_call* b);
/* The batch call against moving opponents (f1l_plan_motion's prediction per scenario): opp_vel
 * [S,max_opp,2] f64 map-frame velocities of b->opp's opponents, v_min as f1l_plan_motion.  Scenario
 * s is bit-identical to f1l_plan_motion on the same inputs (with b->weights: after f1l_set_config
 * with those weights).  F1L_ERR_INVALID_ARG for a non-finite or non-positive v_min, or opp_vel
 * NULL with max_opp > 0.  _dev: device buffers, caller's stream, no sync; every velocity of an
 * opponent in use must be finite (not checked).  Host version: through the chunked pipeline,
 * opp_vel travelling with each chunk's inputs; a non-finite velocity of an opponent in use is
 * F1L_ERR_INVALID_ARG. */
int f1l_plan_batch_motion_dev(f1l_handle h, const f1l_batch_call* b, const double* opp_vel_dev,
                              double v_min, void* stream);
int f1l_plan_batch_motion(f1l_handle h, const f1l_batch_call* b, const double* opp_vel, double v_min);

/*
 * Closed-loop rollouts on the device: a fleet of S kinematic-bicycle cars (f1l_rollout_st_dev below:
 * dynamic single-track cars) advanced n_steps planning
 * steps.  Replaces the user loop around the planner -- plan, then step the vehicle
 * (lattice_planner.py:204-214 plus the gym step of examples/control/pure_pursuit.py:47-57, which
 * is not part of the reference checkout) -- with no host synchronisation and no host copy inside
 * the steps.  Device buffers, caller's stream, no sync.
 *
 * Cars form races of `group` consecutive scenarios [g*group, (g+1)*group); group = 1: independent
 * cars without opponents.  Planning step k, for every car:
 *   1. plan from (x, y, theta, v) exactly as f1l_plan_batch_prev_dev with update_prev = 1 on the
 *      fleet's prev_theta / has_prev; the opponents are the other group-1 cars of the race at their
 *      step-k poses, in race order without the car itself (crashed cars included);
 *   2. steer = clamp(steer_cmd, +-max_steer); target = min(speed_cmd, v_max), or 0 when the plan
 *      had no feasible candidate (best_cost = +inf; sets F1L_CAR_NO_FEASIBLE for this step);
 *   3. `substeps` times, float64: v += clamp(target - v, +-max_accel*dt), x += v cos(theta) dt,
 *      y += v sin(theta) dt, theta += v / wheelbase * tan(steer) dt (wheelbase of the f1l_config;
 *      theta is not wrapped);
 *   4. after every substep, at the new poses: the footprint (car_length x car_width) against the
 *      map with the configured collision_mode (nine probes, or three discs on the distance
 *      transform; out of bounds = occupied; float64, cell = floor((p - origin) / res)) sets
 *      F1L_CAR_HIT_MAP, a float64 SAT against every other car of the race (touching = free) sets
 *      F1L_CAR_HIT_CAR on both.  The hit bits are sticky and freeze the car: it keeps its pose at
 *      v = 0, is still planned and is still an opponent of the others;
 *   5. progress: the nearest raceline segment in a window of 32 segments starting 4 behind the
 *      tracked one (cyclic over the n-1 segments, nearest_point's float64 operations, first
 *      minimum); s = cum[i] + t * len[i]; progress += (s - s_prev) wrapped into [-lap/2, lap/2),
 *      lap = cum[n-1] + |p_0 - p_{n-1}|, so counting continues across the raceline's seam.
 * A car with track_i < 0 at the start of a call is re-acquired by a global nearest_point (its
 * progress stays as given).  All state lives in the fleet buffers: run(30) + run(30) is
 * bit-identical to run(60).  A reset is a caller write: new pose, has_prev = 0, status = 0,
 * track_i = -1.
 */
#define F1L_CAR_HIT_MAP 1u
#define F1L_CAR_HIT_CAR 2u
#define F1L_CAR_NO_FEASIBLE 4u
#define F1L_MAX_GROUP (1 + F1L_MAX_OPP)   /* cars per race */

/* Defaults: dt 0.01, substeps 1, group 1, max_steer 0.4189, max_accel 9.51 (the steering and
 * acceleration limits the closed-loop tests of the batch planner use), v_max +inf. */
typedef struct {
    double dt;           /* integration step (s), > 0 */
    int32_t substeps;    /* integration steps per planning step, >= 1 */
    int32_t group;       /* cars per race, 1..F1L_MAX_GROUP, divides n_scenarios */
    double max_steer;    /* steering limit (rad), > 0 */
    double max_accel;    /* acceleration limit (m/s^2), > 0 */
    double v_max;        /* speed cap (m/s), > 0, may be +inf */
} f1l_rollout_config;

/* The fleet, device buffers read and written in place (S cars, M = n_samples). */
typedef struct {
    double* state;        /* [S,4] x, y, theta, v */
    float* prev_theta;    /* [S,M] previous paths, as f1l_plan_batch_prev_dev */
    uint8_t* has_prev;    /* [S] */
    uint8_t* status;      /* [S] F1L_CAR_* */
    double* progress;     /* [S] metres along the raceline */
    int32_t* track_i;     /* [S] tracked raceline segment, < 0: re-acquire */
    double* track_s;      /* [S] arc length at the tracked point */
} f1l_fleet;

/* Optional per-step record (T = n_steps), each buffer nullable. */
typedef struct {
    double* state;        /* [T,S,4] state at the START of step k */
    double* steer_speed;  /* [T,S,2] raw planner command of step k */
    int32_t* best_idx;    /* [T,S] chosen candidate of step k */
    uint8_t* status;      /* [T,S] status after step k */
    double* progress;     /* [T,S] progress after step k */
} f1l_rollout_trace;

int f1l_default_rollout_config(f1l_rollout_config* rc);

/* F1L_ERR_INVALID_ARG for a null handle, config or fleet pointer, group outside 1..F1L_MAX_GROUP,
 * n_scenarios not a positive multiple of group, substeps < 1, a dt / max_steer / max_accel / v_max
 * that is not positive (NaN included) or n_steps < 0.  n_steps = 0 does nothing.  The handle owns
 * the opponent table ([S,16,3] f64 + [S] i32) and the command scratch; one call in flight per
 * handle.  Numpy users go through the Python layer (Fleet), which copies once per call. */
int f1l_rollout_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_fleet* fleet,
                    int n_scenarios, int n_steps, const f1l_rollout_trace* trace, void* stream);

/* The same with cost weights per car: every step plans car s with weights_dev[s] as
 * f1l_plan_batch_call_dev does.  weights_dev [S,F1L_N_TERMS] f32 device buffer, read only, or
 * NULL: f1l_rollout_dev. */
int f1l_rollout_weights_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_fleet* fleet,
                            const float* weights_dev, int n_scenarios, int n_steps,
                            const f1l_rollout_trace* trace, void* stream);

/*
 * The dynamic single-track (ST) vehicle model of f1tenth_gym (CommonRoad's vehicle_dynamics_st),
 * for rollouts whose cars understeer, slide and answer the steering late.  Defaults are
 * f1tenth_gym's; max_steer, max_accel and v_max stay in f1l_rollout_config.
 */
typedef struct {
    double mu;             /* surface friction coefficient, > 0 */
    double C_Sf;           /* front cornering stiffness coefficient (1/rad), > 0 */
    double C_Sr;           /* rear cornering stiffness coefficient (1/rad), > 0 */
    double lf;             /* centre of gravity to front axle (m), > 0 */
    double lr;             /* centre of gravity to rear axle (m), > 0 */
    double h;              /* height of the centre of gravity (m), >= 0 */
    double m;              /* mass (kg), > 0 */
    double I;              /* yaw moment of inertia (kg m^2), > 0 */
    double max_steer_vel;  /* steering rate limit (rad/s), > 0 */
    double v_switch;       /* speed above which the acceleration limit falls as 1/v (m/s), > 0 */
    double v_kin;          /* speed below which the kinematic form is used (m/s), > 0 */
} f1l_vehicle;

/* Defaults: mu 1.0489, C_Sf 4.718, C_Sr 5.4562, lf 0.15875, lr 0.17145, h 0.074, m 3.74,
 * I 0.04712, max_steer_vel 3.2, v_switch 7.319, v_kin 0.5. */
int f1l_default_vehicle(f1l_vehicle* veh);

/*
 * f1l_rollout_weights_dev with the ST model.  The fleet's state (x, y, psi, v) is unchanged and
 * still what the planner reads (theta = psi, (x, y) the model's reference point, which the
 * footprint, collision tests, progress and opponent table use as before).  dyn_dev [S,3] f64
 * (steering angle delta, yaw rate, slip angle beta) is read and written in place; zeros for a car
 * at rest.  Every rule of f1l_rollout_dev holds except step 3, which becomes, per substep:
 *   sv = clamp((clamp(steer_cmd, +-max_steer) - delta) / dt, +-max_steer_vel);
 *   a = clamp((target - v) / dt, -max_accel, a_pos), a_pos = max_accel * v_switch / v when
 *   v > v_switch, else max_accel (f1tenth_gym's power limit);
 *   with (sv, a) held, one classical RK4 step in float64 of (x, y, delta, v, psi, yaw rate, beta)
 *   under f1tenth_gym's equations: the kinematic form when |v| < v_kin, else the dynamic one
 *   (L = lf + lr, g = 9.81, load transfer through h).  psi is not wrapped.
 * A frozen car keeps its pose and delta at v = yaw rate = beta = 0.
 *
 * The tyres are linear and never saturate, as in f1tenth_gym: there is no friction circle, so the
 * model has no grip limit at high lateral acceleration.  RK4 is stable here only for a small
 * enough dt: the fastest (yaw rate, beta) mode is at the lowest dynamic speed, v = v_kin, where
 * with the defaults and dt = 0.01 it has dt * |lambda| = 2.27, inside RK4's real-axis limit of
 * 2.785.  A larger dt or a smaller v_kin can make the integration diverge.
 *
 * trace_dyn_dev [T,S,3] f64 or NULL: dyn at the START of step k.  F1L_ERR_INVALID_ARG as
 * f1l_rollout_dev, and for a null vehicle or dyn_dev, any of mu, C_Sf, C_Sr, lf, lr, m, I,
 * max_steer_vel, v_switch, v_kin that is not positive (NaN included), or a negative or NaN h.
 */
int f1l_rollout_st_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_vehicle* veh,
                       const f1l_fleet* fleet, double* dyn_dev, const float* weights_dev,
                       int n_scenarios, int n_steps, const f1l_rollout_trace* trace,
                       double* trace_dyn_dev, void* stream);

/*
 * Rollouts whose planners predict their opponents: as f1l_rollout_st_dev (veh != NULL, dyn_dev its
 * state) or f1l_rollout_weights_dev (veh NULL: kinematic bicycle; dyn_dev, trace_dyn_dev ignored),
 * but every step plans through f1l_plan_batch_motion_dev with v_min.  The step kernel writes the
 * next step's opponent velocities next to the opponent table (a [S,F1L_MAX_OPP,2] table the handle
 * owns): v (cos theta, sin theta) for a kinematic car, v (cos(psi + beta), sin(psi + beta)) for a
 * single-track car with slip angle beta, 0 for a frozen car.  F1L_ERR_INVALID_ARG as those calls,
 * and for a non-finite or non-positive v_min.
 */
int f1l_rollout_predict_dev(f1l_handle h, const f1l_rollout_config* rc, const f1l_vehicle* veh,
                            const f1l_fleet* fleet, double* dyn_dev, const float* weights_dev,
                            double v_min, int n_scenarios, int n_steps, const f1l_rollout_trace* trace,
                            double* trace_dyn_dev, void* stream);

/*
 * Batched nearest_point + pure-pursuit lookahead over B poses on the uploaded track.
 * Replaces nearest_point (utils/utils.py:37-67), intersect_point (:69-151), get_actuation
 * (:153-161) and PurePursuitPlanner._get_current_waypoint / plan (pure_pursuit.py:56-122).
 *   poses [B,3] f64 (x, y, theta)
 * outputs (any may be NULL):
 *   nearest [B,4] f64 = (proj_x, proj_y, dist, t);  nearest_i [B] i32
 *   lookahead [B,4] f64 = (p_x, p_y, t2, found);    lookahead_i [B] i32 (un-modded, may be -1)
 *   actuation [B,2] f64 = (steer, speed);           status [B] i32 (1 intersect branch,
 *                                                   2 reacquire branch, 0 no lookahead point)
 */
int f1l_pure_pursuit_batch_dev(f1l_handle h, const double* poses_dev, int n_poses,
                               double lookahead_distance, double* nearest_dev,
                               int32_t* nearest_i_dev, double* lookahead_dev,
                               int32_t* lookahead_i_dev, double* actuation_dev,
                               int32_t* status_dev, void* stream);
int f1l_pure_pursuit_batch(f1l_handle h, const double* poses, int n_poses,
                           double lookahead_distance, double* nearest, int32_t* nearest_i,
                           double* lookahead, int32_t* lookahead_i, double* actuation,
                           int32_t* status);

/*
 * Front-axle tracking errors for B vehicle states on the uploaded track: the nearest_point
 * consumer shared by the Stanley and LQR controllers.  Replaces StanleyPlanner.calc_theta_and_ef
 * + controller (control/stanley/stanley.py:57-112) and LQRPlanner.calc_control_points
 * (control/lqr/lqr.py:60-102).
 *   poses [B,4] f64 (x, y, theta, velocity)
 *   front [B,6] f64 = (theta_e, ef, theta_raceline, kappa_ref, goal_velocity,
 *                      delta = atan2(k_path * ef, velocity) + theta_e)
 *   nearest_i [B] i32 (target_index) or NULL
 */
int f1l_front_axle_batch_dev(f1l_handle h, const double* poses_dev, int n_poses, double wheelbase,
                             double k_path, double* front_dev, int32_t* nearest_i_dev,
                             void* stream);
int f1l_front_axle_batch(f1l_handle h, const double* poses, int n_poses, double wheelbase,
                         double k_path, double* front, int32_t* nearest_i);

/* intersect_point (utils/utils.py:69-151) for B independent queries on the uploaded track:
 * points [B,2], radius, start parameter t [B]; out [B,4] = (p_x, p_y, t, found), out_i [B].
 * Every t must lie in [0, N) (N waypoints): anything else, NaN included, is F1L_ERR_INVALID_ARG
 * (the reference indexes waypoint int(t) unchecked). */
int f1l_intersect_point_batch(f1l_handle h, const double* points, const double* t_start,
                              int n, double radius, int wrap, double* out, int32_t* out_i);

/* get_actuation (utils/utils.py:153-161) for B queries: in [B,7] = (pose_theta, lp_x, lp_y,
 * lp_speed, pos_x, pos_y, lookahead_distance); out [B,2] = (speed, steer) in the reference's
 * return order. */
int f1l_get_actuation_batch(f1l_handle h, const double* in, int n, double wheelbase,
                            double* out);

/* Work counters of the deviation pass are collected only while switched on (default off: the
 * counting costs every CTA of eval_kernel a barrier and two global atomics). */
int f1l_set_stats(f1l_handle h, int on);
/* Work counters of the deviation pass since the last call (synchronises the handle's stream and
 * resets them): out[0] = (candidate, window segment) pairs evaluated, out[1] = candidates that
 * reached the pass (valid trajectories).  With prune_window = 0, out[0] / out[1] is the padded
 * window length.  n >= 2. */
int f1l_get_stats(f1l_handle h, uint64_t* out, int n);

/* Which eval_kernel<IPL, S, SG, NW, MINB, PW> instance the last f1l_plan* call launched and its
 * CTA plan: out[0..4] = IPL, S, SG, NW (warps per CTA), MINB (resident CTAs per SM asked of the
 * compiler); out[5] = candidates per CTA, out[6] = CTAs per scenario, out[7] = candidates a warp
 * solves together (4 = shared Newton).  n >= 8.  With n >= 10 also out[8] = 1 on the persistent
 * grid of a lone dense query and out[9] = PW (1: per-scenario cost weights); with n >= 11
 * out[10] = MO (1: the moving-opponent twin of the PW instance, f1l_plan_motion and friends).
 * Evidence for bench.py / profiles. */
int f1l_last_eval_shape(f1l_handle h, int32_t* out, int n);

/* Timing / evidence helpers: number of kernels launched by this handle so far, and the device
 * time (ms, CUDA events on the handle's stream) of the kernels of the last host-pointer call. */
int64_t f1l_launch_count(f1l_handle h);
/* The single-query chain (input copy, sampler, eval, select, result copy) is replayed as one CUDA
 * graph, re-captured when an upload / configuration change or the requested outputs change a
 * kernel argument.  on = 0 falls back to plain stream launches (default: on). */
int f1l_set_graph(f1l_handle h, int on);
/* on != 0: f1l_plan* record CUDA events around their three kernels (read with
 * f1l_last_kernel_ms); off by default to keep the single-query latency minimal. */
int f1l_set_timing(f1l_handle h, int on);
/* Mean device time (ms) of the three kernels over the pipeline launches recorded since the last
 * f1l_set_timing call (ring of the most recent 64), and how many launches that covers. */
int f1l_mean_kernel_ms(f1l_handle h, float* sample_ms, float* eval_ms, float* select_ms,
                       int* n_launches);
int f1l_last_kernel_ms(f1l_handle h, float* sample_ms, float* eval_ms, float* select_ms);

/* Host placement for multi-GPU batches (one process per GPU): sets the calling thread's CPU
 * affinity to the CPUs of the NUMA node the device's PCIe root hangs off (sysfs), so that pinned
 * host buffers allocated afterwards are first-touched on that node and the result copies of the
 * ranks do not all cross the socket interconnect.  Returns the node (>= 0), -100 when the platform
 * exposes no NUMA placement (nothing changed), or F1L_ERR_NO_DEVICE.  No handle needed. */
int f1l_bind_host_numa(int device);

/* FP32 FMA / MUFU pipe peak microbenchmarks (roofline denominators, SURVEY 8d):
 * returns achieved TFLOP/s (FMA = 2 FLOP) and MUFU Gop/s on the handle's device. */
int f1l_measure_peaks(f1l_handle h, double* fp32_tflops, double* mufu_gops);
/* Extended probes: out[0] FFMA TFLOP/s, out[1] MUFU Gop/s, out[2] packed FFMA2 (fma.rn.f32x2)
 * TFLOP/s, out[3] warp-instructions per clock per SM of an FFMA + FMNMX mix (n >= 4). */
int f1l_measure_peaks_ex(f1l_handle h, double* out, int n);

/* Host-side launch planning, callable without a device (tests of the host logic):
 * f1l_debug_eval_plan: the CTA plan of eval_kernel for n_scenarios queries of n_cand candidates
 * and M arc samples on sm_count SMs -- out[0] = warps per CTA, out[1] = candidates per CTA,
 * out[2] = CTAs per scenario, out[3] = candidates a warp solves together (n >= 4).  This is the
 * plan of a batch call without per-scenario weights; f1l_debug_eval_choice with flags 0 gives the
 * same four entries.
 * f1l_debug_eval_choice: the eval_kernel instance and CTA plan a pipeline launch chooses.  flags:
 * F1L_EVAL_LONE for a single query (f1l_plan*, n_scenarios = 1: persistent grid and wide build
 * allowed), F1L_EVAL_WEIGHTS for a call with per-scenario cost weights.  out[0..3] as above (on
 * the persistent grid out[2] is its CTA count and out[3] the candidates per pull); with n >= 12
 * also the bucket's out[4] = largest M, out[5] = IPL, out[6] = S, out[7] = SG, then out[8] = MINB
 * of the chosen build (0: not built), out[9] = 1 for the wide build, out[10] = 1 for the
 * persistent grid, out[11] = PW; with n >= 13 out[12] = the largest window (segments) the build's
 * shared memory holds.
 * f1l_debug_eval_builds: every row of the instance table, 8 entries each: largest M, IPL, S, SG,
 * then MINB of the 4-, 7- and 8-warp builds and of the wide build (0: not built).  Every build
 * but the wide one also has its PW twin.  Returns the number of rows (n >= 8 x rows).
 * f1l_debug_pp_parts: into how many parts pp_scan_kernel splits a track of n_waypoints for
 * n_poses poses when `slots` one-warp CTAs are resident on the device (> 0), or an error (< 0). */
#define F1L_EVAL_LONE 1
#define F1L_EVAL_WEIGHTS 2
int f1l_debug_eval_plan(int n_cand, int n_scenarios, int M, int sm_count, int generator,
                        int32_t* out, int n);
int f1l_debug_eval_choice(int n_cand, int n_scenarios, int M, int sm_count, int generator, int flags,
                          int32_t* out, int n);
int f1l_debug_eval_builds(int32_t* out, int n);
int f1l_debug_pp_parts(int n_poses, int n_waypoints, int slots);

/* Debug / test hook: the float32 per-query constants of the last f1l_plan* call, for
 * teacher-forced collision checks.  out_f[72]: cos, sin of the pose heading; grid transform A00
 * A01 A10 A11 fx fy; then 16 opponents x (x, y, cos, sin) in the vehicle frame.  out_i[6]: grid
 * ix0, iy0, nearest segment, window start, window length, opponent count. */
int f1l_debug_query_ctx(f1l_handle h, float* out_f, int32_t* out_i);

/* Debug / test hook: the float32 motion constants of the last f1l_plan_motion call, for
 * teacher-forced collision checks: out[0] = k_t, out[1 + 2k], out[2 + 2k] = opponent k's velocity
 * (wx, wy) in the vehicle frame (0 for unused slots).  n >= 1 + 2 F1L_MAX_OPP. */
int f1l_debug_motion_ctx(f1l_handle h, float* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* F1L_H */
