"""Drop-in for f1tenth_planning/planning/lattice_planner/lattice_planner.py:40-296.

Same class, constructor, plug-in hooks and ``plan`` 3-tuple as the reference; underneath, the
goal-grid sampler, cubic-spiral generation, fused cost + collision stage and argmin run as
sm_100a CUDA kernels through the C-ABI library (include/f1l.h).

Reference-compatible surface
    LatticePlanner(wheelbase=0.33, waypoints=None)                      :44
    .add_cost_function(func | [funcs])                                  :57-75
    .add_sample_function(func)                                          :77-98
    .add_selection_function(func)                                       :100-111
    .sample(pose_x, pose_y, pose_theta, velocity, waypoints)            :113-128
    .eval(all_traj, cost_weights)                                       :130-156
    .select(all_costs)                                                  :159-172
    .plan(pose_x, pose_y, pose_theta, velocity, waypoints=None)         :174-214
        -> (steering_angle, speed, selected_traj [M,4])
    sample_lookahead_square(...), get_length_cost(...) ...              :223-296

Additive (north-star) surface
    .plan(..., opponent_poses=[K,3])      opponents in the map frame
    .plan_detailed(...) / .last           PlanDetail: best_idx, costs[C], terms[C,5], flags[C] ...
    .plan_batch(poses[S,4], opponents[S,K,3], n_opp[S][, prev_theta=[S,M], has_prev=[S],
                update_prev=True])  per-scenario previous paths, carried in place step to step
    .rollout(poses[S,4], n_steps, group=1, weights=None, vehicle=None, **kw)
                                         closed-loop rollouts of a fleet on the device
    .set_map(occupancy, origin, resolution), .set_goal_grid(lookaheads, widths)

With no plug-ins registered every stage runs on the GPU.  A registered ``sample_func`` replaces
only the sampler (its goals are uploaded); registered ``cost_funcs`` are user Python code and are
evaluated on the host over GPU-generated trajectories, as the reference's ``eval`` does.
"""

import numpy as np

from .engine import (Engine, PlanDetail, FLAG_VALID, FLAG_COLLIDE_OPP, FLAG_COLLIDE_MAP,  # noqa: F401
                     fingerprint)
from .pure_pursuit import PurePursuitPlanner
from . import synth

# constants the reference's cost helpers reference but never define (lattice_planner.py:277-294)
NUM_STEPS = 100
N_SHIFT = 5
N_CULL = 10


class LatticePlanner():
    """Sampling lattice planner (reference lattice_planner.py:40)."""

    def __init__(self, wheelbase=0.33, waypoints=None, device=None, **config):
        self.wheelbase = wheelbase
        self.waypoints = waypoints

        self.sample_func = None
        self.cost_funcs = []
        self.selection_func = None
        self.cost_weights = None   # weights for registered python cost functions (eval)

        # :55 (default wheelbase, as upstream).  Kept for API parity; plan() tracks on the device
        # (select_kernel), also for user-selected candidates
        self.tracker = PurePursuitPlanner(device=device)

        self._device = device
        config.setdefault("wheelbase", float(wheelbase))
        self._config = config
        self._engine = None
        self._key = None
        self._lookaheads = synth.DEFAULT_LOOKAHEADS.copy()   # :228
        self._widths = synth.DEFAULT_WIDTHS.copy()           # :229
        self._grid_dirty = True
        self._map = None
        self._shard = None         # (rank, world) after shard_across()
        self.last = None

    # -- reference plug-in API ------------------------------------------------------------------
    def add_cost_function(self, func):
        """lattice_planner.py:57-75"""
        if type(func) is list:
            self.cost_funcs.extend(func)
        else:
            self.cost_funcs.append(func)

    def add_sample_function(self, func):
        """lattice_planner.py:77-98; func(pose_x, pose_y, pose_theta, velocity, waypoints) ->
        goal_grid [N,3] in the vehicle frame."""
        self.sample_func = func

    def add_selection_function(self, func):
        """lattice_planner.py:100-111; func(costs) -> index."""
        self.selection_func = func

    def sample(self, pose_x, pose_y, pose_theta, velocity, waypoints):
        """lattice_planner.py:113-128"""
        if self.sample_func is None:
            raise NotImplementedError('Please set a sample function before sampling.')
        goal_grid = self.sample_func(pose_x, pose_y, pose_theta, velocity, waypoints)
        return goal_grid

    def eval(self, all_traj, cost_weights):
        """lattice_planner.py:130-156 (user cost functions, host)."""
        if len(self.cost_funcs) == 0:
            raise NotImplementedError('Please set cost functions before evaluating.')
        if len(self.cost_funcs) != len(cost_weights):
            raise ValueError('Length of cost weights must be the same as number of cost functions.')
        if np.sum(cost_weights) != 1:
            raise ValueError('Cost weights must add up to 1.')
        all_costs = []
        for traj in all_traj:
            cost = 0.
            for i, func in enumerate(self.cost_funcs):
                cost += cost_weights[i] * func(traj)
            all_costs.append(cost)
        return all_costs

    def select(self, all_costs):
        """lattice_planner.py:159-172"""
        if self.selection_func is None:
            self.selection_func = np.argmin
        best_idx = self.selection_func(all_costs)
        return best_idx

    # -- additive configuration -----------------------------------------------------------------
    def set_goal_grid(self, lookahead_distances, widths):
        self._lookaheads = np.asarray(lookahead_distances, dtype=np.float64).ravel()
        self._widths = np.asarray(widths, dtype=np.float64).ravel()
        self._grid_dirty = True

    def set_map(self, occupancy, origin, resolution):
        """uint8 occupancy [H,W] (0 free), origin (x, y) of cell (0,0), metres per cell."""
        self._map = (np.ascontiguousarray(occupancy, dtype=np.uint8), tuple(origin), float(resolution))
        if self._engine is not None:
            self._engine.set_grid(*self._map)

    def load_map(self, yaml_path):
        """ROS map_server yaml + image (examples/control/Spielberg_map.yaml) -> set_map"""
        from . import io
        self.set_map(*io.load_map(yaml_path))

    def configure(self, **config):
        self._config.update(config)
        if self._engine is not None:
            self._engine.configure(**config)

    @property
    def engine(self):
        return self._sync()

    def _sync(self):
        if self.waypoints is None:
            raise ValueError('Please set waypoints during planner instantiation or when calling plan()')
        if self._engine is None:
            self._engine = Engine(device=self._device, **self._config)
            if self._map is not None:
                self._engine.set_grid(*self._map)
        # Has the raceline changed?  Every element takes part in the fingerprint (in-place edits of
        # single rows are detected), ~8 us per call.
        wp = self.waypoints
        arr = wp if isinstance(wp, np.ndarray) else np.asarray(wp, dtype=np.float64)
        key = fingerprint(arr)
        if key != self._key:
            w = np.ascontiguousarray(arr, dtype=np.float64)
            if w.ndim != 2 or w.shape[1] < 4:
                raise ValueError('Waypoints needs to be a (Nxm), m >= 4 (x, y, v, psi[, kappa]), numpy array!')
            self._engine.set_track(w)
            self._key = key
        if self._grid_dirty:
            self._engine.set_goal_grid(self._lookaheads, self._widths)
            self._grid_dirty = False
        return self._engine

    # -- one dense query across the GPUs of a node --------------------------------------------------
    def shard_across(self, group=None):
        """Collective over a torch.distributed group (one process per GPU): from now on plan() /
        plan_detailed() evaluate only this rank's lookahead rows (rank, rank + world, ...) and the
        ranks' minima meet inside the select kernel over NVLink peer memory, so every rank returns
        the global winner.  Every rank must then call plan() with the same arguments.  Queries
        that run user plug-ins (sample / cost / selection functions) stay unsharded."""
        import torch.distributed as dist
        eng = self._sync()
        eng.attach_peers(group)
        self._shard = (dist.get_rank(group), dist.get_world_size(group))

    def unshard(self, group=None):
        if self._shard is not None and self._engine is not None:
            self._engine.detach_peers(group)
        self._shard = None

    # -- planning -------------------------------------------------------------------------------
    def plan_detailed(self, pose_x, pose_y, pose_theta, velocity, waypoints=None,
                      opponent_poses=None, want_states=False, want_map=False, opponent_velocities=None):
        """Full result of one query as a PlanDetail (see engine.PlanDetail).  want_map adds
        ``best_traj_map`` [M,4] = (X, Y, v, Theta), the best trajectory in the map frame with a
        speed column (what a map-frame tracker consumes, SURVEY B.8).  opponent_velocities [K,2]
        (vx, vy) m/s, map frame: plan against the opponents' constant-velocity prediction
        (Engine.plan; not with a user sampler or a row shard)."""
        if waypoints is not None:
            self.waypoints = waypoints
        eng = self._sync()
        pose = np.array([pose_x, pose_y, pose_theta, velocity], dtype=np.float64)
        custom_cost = len(self.cost_funcs) > 0
        custom_select = self.selection_func is not None and self.selection_func is not np.argmin
        plugins = custom_cost or custom_select
        need_states = want_states or custom_cost
        if opponent_velocities is not None and (self.sample_func is not None or self._shard is not None):
            raise ValueError("opponent_velocities cannot be combined with a user sampler or a row shard")
        if opponent_velocities is not None:
            d = eng.plan(pose, opponent_poses, want_states=need_states, want_map=want_map and not plugins,
                         opponent_velocities=opponent_velocities)
        elif self.sample_func is not None:
            goal_grid = np.asarray(self.sample(pose_x, pose_y, pose_theta, velocity, self.waypoints),
                                   dtype=np.float64).reshape(-1, 3)
            d = eng.plan_goals(pose, goal_grid, opponent_poses, want_states=need_states,
                               want_map=want_map and not plugins)
        elif self._shard is not None and not (need_states or plugins):
            d = eng.plan(pose, opponent_poses, rows=self._shard, want_map=want_map)
        else:
            d = eng.plan(pose, opponent_poses, want_states=need_states,
                         want_map=want_map and not plugins)
        if plugins:
            # User python plug-ins (lattice_planner.py:130-172) run on the host over the
            # GPU-generated trajectories; candidates the GPU found invalid or in collision keep
            # cost +inf whatever the user functions say.  The chosen candidate then goes back to
            # the device, which regenerates it and runs the same tracker as the built-in
            # selection (f1l_select_candidate) -- same frame, speed column, literal_tracker,
            # wheelbase and max_reacquire, and it becomes the next call's previous path.
            bad = ((d.flags & FLAG_VALID) == 0) | ((d.flags & (FLAG_COLLIDE_OPP | FLAG_COLLIDE_MAP)) != 0)
            if custom_cost:
                all_traj = d.states.astype(np.float64)
                all_traj[:, :, 3] = np.abs(all_traj[:, :, 3])   # utils.py:293 column = |kappa|
                weights = self.cost_weights
                if weights is None:
                    weights = [1.0 / len(self.cost_funcs)] * len(self.cost_funcs)
                costs = np.asarray(self.eval(all_traj, weights), dtype=np.float64)
                costs[bad] = np.inf
            else:
                costs = d.costs.astype(np.float64)
            idx = int(self.select(costs))
            t = eng.select_candidate(idx, costs[idx], update_prev=True, want_map=want_map)
            d = d._replace(steer=t.steer, speed=t.speed, best_traj=t.best_traj, best_idx=idx,
                           best_cost=float(costs[idx]), costs=costs.astype(np.float32),
                           no_feasible=t.no_feasible, tracker_found=t.tracker_found,
                           best_traj_map=t.best_traj_map)
        self.last = d
        return d

    def rollout(self, poses, n_steps, group=1, weights=None, vehicle=None, **kw):
        """Closed-loop rollouts on the device for host users: the cars at `poses` [S,4] (x, y,
        theta, v), raced in groups of `group` consecutive cars, each planned with its row of
        `weights` [S,5] (None: the configured weights), advanced n_steps planning steps
        (keywords as rollout.Fleet.run).  Returns the per-step RolloutTrace as numpy arrays and the
        final (state [S,4], status [S], progress [S]).  With a rollout.Vehicle the cars follow the
        single-track model: the trace is a SingleTrackTrace and the final tuple ends with dyn [S,3]."""
        fleet = self._sync().fleet(poses, group, weights, vehicle)
        tr = fleet.run(n_steps, trace=True, **kw)
        trace = type(tr)(*(t.cpu().numpy() for t in tr))
        final = (fleet.state.cpu().numpy(), fleet.status.cpu().numpy(), fleet.progress.cpu().numpy())
        return trace, final + ((fleet.dyn.cpu().numpy(),) if vehicle is not None else ())

    def plan(self, pose_x, pose_y, pose_theta, velocity, waypoints=None, opponent_poses=None,
             opponent_velocities=None):
        """lattice_planner.py:174-214 -> (steering_angle, speed, selected_traj [M,4]).

        selected_traj columns are (x, y, theta, |kappa|) in the vehicle frame like
        utils.sample_traj (utils/utils.py:285-295); the signed-curvature float32 trajectory,
        index, cost vector and flags are in ``self.last``."""
        d = self.plan_detailed(pose_x, pose_y, pose_theta, velocity, waypoints, opponent_poses,
                               opponent_velocities=opponent_velocities)
        traj = d.best_traj.astype(np.float64)
        traj[:, 3] = np.abs(traj[:, 3])
        return d.steer, d.speed, traj

    def plan_batch(self, poses, opponents=None, n_opp=None, **kw):
        """S independent scenarios: poses [S,4], opponents [S,K,3], n_opp [S] -> BatchPlan
        (best_idx [S], best_cost [S], best_traj [S,M,4], costs [S,C], flags, steer_speed [S,2]).

        Each scenario may carry its own previous path for the similarity cost, the batched form
        of what plan() keeps from call to call: prev_theta [S,M] float32 (C-contiguous) and
        has_prev [S] bool / uint8.  With update_prev=True both are overwritten in place with this
        step's best trajectories' theta columns and ones, so a loop of S cars passes them back
        unchanged on the next step.  weights [S,5] gives each scenario its own cost weights and
        want_terms=True returns the per-term costs [S,C,5] as BatchPlan.terms.  Keywords go to
        Engine.plan_batch."""
        return self._sync().plan_batch(poses, opponents, n_opp, **kw)


# ---------------------------------------------------------------------------------------------
# example sampler / cost helpers with the reference's names
# ---------------------------------------------------------------------------------------------
_sampler_planners = {}


def sample_lookahead_square(pose_x, pose_y, pose_theta, velocity, waypoints,
                            lookahead_distances=[0.4, 0.6, 0.8, 1.0],
                            widths=np.linspace(-1.0, 1.0, num=7)):
    """Goal grid around look-ahead points on the raceline (lattice_planner.py:223-260, with the
    repairs listed in DESIGN.md: every centre gets every width, offsets along the raceline
    normal, goals in the vehicle frame).  Runs the GPU sampler; returns [n_L*n_W, 3]."""
    w = np.ascontiguousarray(waypoints, dtype=np.float64)
    key = fingerprint(w)
    pl = _sampler_planners.get("p")
    if pl is None:
        pl = LatticePlanner()
        _sampler_planners["p"] = pl
    if _sampler_planners.get("key") != key:
        pl.waypoints = w
        _sampler_planners["key"] = key
    pl.set_goal_grid(lookahead_distances, widths)
    eng = pl._sync()
    d = eng.plan(np.array([pose_x, pose_y, pose_theta, velocity], dtype=np.float64),
                 update_prev=False)
    return d.goals.astype(np.float64)


def get_length_cost(param_list):
    """lattice_planner.py:268-271"""
    return 1. / param_list[:, 0]


def get_max_curvature(traj_list, num_traj):
    """lattice_planner.py:273-278 (NUM_STEPS defined here)"""
    return np.max(np.abs(traj_list[:num_traj * NUM_STEPS, 3].reshape(num_traj, NUM_STEPS)), axis=1)


def get_mean_curvature(traj_list, num_traj):
    """lattice_planner.py:280-285"""
    return np.mean(np.abs(traj_list[:num_traj * NUM_STEPS, 3].reshape(num_traj, NUM_STEPS)), axis=1)


def get_similarity_cost(traj_list, prev_path, num_traj):
    """lattice_planner.py:287-296"""
    prev_shifted = prev_path[N_SHIFT:-N_CULL, 2]
    th = traj_list[:num_traj * NUM_STEPS, 2].reshape(num_traj, NUM_STEPS)
    return np.sum(np.square(th[:, :-N_SHIFT - N_CULL] - prev_shifted[None, :]), axis=1)
