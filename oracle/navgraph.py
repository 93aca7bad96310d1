"""float64 numpy restatement of the GraphMPE ``navigation_graph`` hot path, batched
over envs (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py).

Every function cites the reference lines it follows (paths relative to
the original project's root).  Arithmetic is float64 in the reference's own operation order,
so that this file agrees with the imported reference to ~1e-13
(tests/test_oracle_vs_golden.py pins it against tests/golden/*.npz, which were
produced by running the UNMODIFIED reference: oracle/make_golden.py).

Entity order is the reference's ``World.entities`` (core.py:186):
agents 0..N-1, landmarks N..2N-1, obstacles 2N..2N+O-1, walls 2N+O..2N+O+W-1.

Also restated: walls (``num_walls`` 1 or 2; core.py:36-55, :407-462) and ``graph_feat_type='global'``.
"""
from __future__ import annotations

from dataclasses import dataclass, field, fields
from typing import Dict, Optional

import numpy as np

from . import lexifair as _lexifair
from .philox import philox4x32_10, u01_24

INFO_KEYS = (
    "individual_reward", "Dist_to_goal", "Time_req_to_goal", "Num_agent_collisions",
    "Num_obst_collisions", "Distance_mean", "Distance_variance", "Mean_by_variance",
    "Dists_traveled", "Time_taken", "Time_mean", "Time_stddev", "Time_mean_by_stddev",
    "Min_time_to_goal",
)


@dataclass
class NavConfig:
    """The argparse fields ``Scenario.make_world`` reads (navigation_graph.py:94-129, :144,
    :188, :208) plus the World constants (core.py:153-160, :68, :85; environment.py:307)."""
    num_agents: int = 3
    num_obstacles: int = 3
    world_size: float = 2.0
    max_speed: float = 2.0
    collision_rew: float = 5.0
    goal_rew: float = 5.0
    min_dist_thresh: float = 0.05
    episode_length: int = 25
    fair_rew: float = 1.0
    zeroshift: float = 5.0
    max_edge_dist: float = 1.0
    collaborative: bool = False
    # True  -> navigation_graph.py (FA+FR: tanh fairness term in the reward, :806-823)
    # False -> nav_graph_goalassign_noFair.py (FA: same file minus that term)
    fairness_reward: bool = True
    # 'relative': ego-relative 11-dim node features (:1079-1124);  'global': 7-dim absolute features (:1058-1077)
    graph_feat_type: str = "relative"
    # walls (navigation_graph.py:181-196, :287-324; core.py:36-55, :407-462): 0, 1 or 2 axis-aligned segments of
    # width 0.1 at +-axis, half-length wall_len, orientation redrawn every episode; pinned by tests/golden/n3_o3_w2.npz
    # and n4_o2_w1.npz (the wall instantiations of the group-per-env kernels are held to the same fixtures).
    num_walls: int = 0
    wall_width: float = 0.1
    wall_contact_force: float = 2.2e2
    wall_contact_margin: float = 2.4e-2
    dt: float = 0.1
    damping: float = 0.25
    contact_force: float = 3e2
    contact_margin: float = 2e-2
    entity_size: float = 0.05
    sensitivity: float = 5.0
    mass: float = 1.0

    @property
    def num_entities(self) -> int:
        return 2 * self.num_agents + self.num_obstacles + self.num_walls

    @property
    def node_feat_dim(self) -> int:
        return 11 if self.graph_feat_type == "relative" else 7


STATE_FIELDS = ("pos", "vel", "p_dist", "landmark_pos", "obstacle_pos", "goal_match",
                "dists_to_goal", "times_required", "dist_left_to_goal",
                "num_agent_collisions", "num_obstacle_collisions",
                "dist_traveled_mean", "dist_traveled_stddev", "step", "min_time", "episode")


@dataclass
class NavState:
    """Everything ``World`` + ``Scenario`` carry between steps (SURVEY.md section 7)."""
    pos: np.ndarray                      # [B,N,2]
    vel: np.ndarray                      # [B,N,2]
    p_dist: np.ndarray                   # [B,N]   core.py:354
    landmark_pos: np.ndarray             # [B,N,2]
    obstacle_pos: np.ndarray             # [B,O,2]
    goal_match: np.ndarray               # [B,N] int   navigation_graph.py:558
    dists_to_goal: np.ndarray            # [B,N]   world.dists_to_goal, -1 = not yet visited
    times_required: np.ndarray           # [B,N]   world.times_required, -1 = not reached
    dist_left_to_goal: np.ndarray        # [B,N]
    num_agent_collisions: np.ndarray     # [B,N]
    num_obstacle_collisions: np.ndarray  # [B,N]
    dist_traveled_mean: np.ndarray       # [B]     world.dist_traveled_mean (carried over resets)
    dist_traveled_stddev: np.ndarray     # [B]
    step: np.ndarray                     # [B] int  env.current_step == world.current_time_step
    min_time: np.ndarray                 # [B,N]   agent.goal_min_time
    episode: np.ndarray                  # [B] int  number of resets so far (RNG counter)
    # walls (None when num_walls == 0)
    wall_axis: Optional[np.ndarray] = None    # [B,W]  wall.axis_pos (navigation_graph.py:288-289, :308)
    wall_orient: Optional[np.ndarray] = None  # [B,W] int  0 = 'H', 1 = 'V' (:298)
    wall_len: Optional[np.ndarray] = None     # [B]    scenario.wall_length = half-length (:183-185, :307)

    def copy(self) -> "NavState":
        return NavState(**{f.name: (None if getattr(self, f.name) is None else getattr(self, f.name).copy())
                           for f in fields(self)})


def _norm2(d):
    """sqrt(dx*dx + dy*dy) -- np.linalg.norm(axis=2) / np.sqrt(np.sum(np.square(.)))
    (core.py:226, navigation_graph.py:583-584)."""
    return np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])


def collision_dist_min(cfg: NavConfig) -> float:
    """``1.05*(size_a + size_b)`` (navigation_graph.py:655, :695, :704, :713)."""
    return 1.05 * (cfg.entity_size + cfg.entity_size)


class NavGraphOracle:
    """B independent navigation_graph envs with the reference's semantics.

    ``seed``/``env_offset`` key the Philox reset stream by *global* env index.
    """

    def __init__(self, cfg: NavConfig, num_envs: int, seed: int = 0, env_offset: int = 0):
        self.cfg = cfg
        self.B = int(num_envs)
        self.seed = int(seed)
        self.env_offset = int(env_offset)
        N, O, B = cfg.num_agents, cfg.num_obstacles, self.B
        z = np.zeros
        self.s = NavState(
            pos=z((B, N, 2)), vel=z((B, N, 2)), p_dist=z((B, N)), landmark_pos=z((B, N, 2)),
            obstacle_pos=z((B, O, 2)),
            # make_world: goal_match_index = arange(N) (navigation_graph.py:93)
            goal_match=np.tile(np.arange(N), (B, 1)),
            dists_to_goal=-np.ones((B, N)), times_required=-np.ones((B, N)),
            dist_left_to_goal=-np.ones((B, N)), num_agent_collisions=z((B, N)),
            num_obstacle_collisions=z((B, N)), dist_traveled_mean=z(B), dist_traveled_stddev=z(B),
            step=z(B, dtype=np.int64), min_time=np.full((B, N), np.inf), episode=z(B, dtype=np.int64))
        if cfg.num_walls:
            if cfg.num_walls > 2:
                raise ValueError("navigation_graph places at most 2 walls (wall_axis has two entries, :289)")
            self.s.wall_axis = z((B, cfg.num_walls))
            self.s.wall_orient = z((B, cfg.num_walls), dtype=np.int64)
            # scenario.wall_length = U(0.2, 0.8) * world_size / 4, drawn once in make_world (:183-185): one Philox
            # draw per env under the reserved episode key 0xFFFFFFFF
            g = (np.arange(B) + self.env_offset).astype(np.uint64)
            r0, _, _, _ = philox4x32_10(
                np.zeros(B, np.uint32), np.full(B, 0xFFFFFFFF, np.uint32), (g & np.uint64(0xFFFFFFFF)).astype(np.uint32),
                (g >> np.uint64(32)).astype(np.uint32), np.uint32(self.seed & 0xFFFFFFFF), np.uint32((self.seed >> 32) & 0xFFFFFFFF))
            u = u01_24(r0)
            self.s.wall_len = ((np.float32(0.2) + np.float32(0.6) * u) * np.float32(cfg.world_size / 4)).astype(np.float64)
        self.last_info: Optional[Dict[str, np.ndarray]] = None

    # ------------------------------------------------------------------ state access
    def get_state(self) -> NavState:
        return self.s.copy()

    def set_state(self, state: NavState) -> None:
        """Inject a state (float64 copies; ints stay ints)."""
        d = {}
        for f in fields(NavState):
            if getattr(state, f.name) is None:
                d[f.name] = None
                continue
            a = np.asarray(getattr(state, f.name))
            if f.name in ("goal_match", "step", "episode", "wall_orient"):
                d[f.name] = a.astype(np.int64).copy()
            else:
                d[f.name] = a.astype(np.float64).copy()
        self.s = NavState(**d)

    # ------------------------------------------------------------------ physics
    def _action_u(self, actions=None, onehot=None) -> np.ndarray:
        """environment.py:265-324 (_set_action, discrete_action_space branch :301-311):
        u = [a1 - a2, a3 - a4] * sensitivity(5.0)."""
        if onehot is None:
            onehot = np.eye(5)[np.asarray(actions, dtype=np.int64)]        # graph_mpe_runner.py:429-431
        oh = np.asarray(onehot, dtype=np.float64)
        u = np.zeros(oh.shape[:-1] + (2,))
        u[..., 0] += oh[..., 1] - oh[..., 2]
        u[..., 1] += oh[..., 3] - oh[..., 4]
        u *= self.cfg.sensitivity
        return u

    def _wall_pos(self) -> np.ndarray:
        """wall.state.p_pos (navigation_graph.py:309-324): the midpoint, (0, axis) for 'H', (axis, 0) for 'V'."""
        s = self.s
        horiz = s.wall_orient == 0
        return np.stack([np.where(horiz, 0.0, s.wall_axis), np.where(horiz, s.wall_axis, 0.0)], axis=-1)   # [B,W,2]

    def _entity_pos(self) -> np.ndarray:
        s = self.s
        parts = [s.pos, s.landmark_pos, s.obstacle_pos]
        if self.cfg.num_walls:
            parts.append(self._wall_pos())               # core.py:186: walls come last in world.entities
        return np.concatenate(parts, axis=1)             # [B,E,2]

    def _forces(self, u: np.ndarray) -> np.ndarray:
        """core.py:277-298 (apply_action_force) + :301-316 (apply_environment_force) +
        :370-404 (get_entity_collision_force, cached-distance branch: dist_min = size_a+size_b)."""
        cfg = self.cfg
        N, E = cfg.num_agents, cfg.num_entities
        ent = self._entity_pos()
        F = cfg.mass * u + 0.0                                   # core.py:291-293 (noise = 0.0)
        k = cfg.contact_margin
        W, O = cfg.num_walls, cfg.num_obstacles
        size = np.full(E, cfg.entity_size)
        if W:
            size[E - W:] = cfg.wall_width                        # Wall.size = width (core.py:48-49): a circle at its midpoint
        for a in range(E):
            a_agent = a < N
            a_collide = a_agent or a >= 2 * N                    # landmarks: collide=False (:169)
            for b in range(a + 1, E):
                b_agent = b < N
                b_collide = b_agent or b >= 2 * N
                if not (a_collide and b_collide):
                    continue                                     # core.py:373-374
                if not (a_agent or b_agent):
                    continue                                     # core.py:375-376
                dist_min = size[a] + size[b]                     # core.py:215
                delta = ent[:, a] - ent[:, b]                    # cached_dist_vect[ia, ib], core.py:222
                dist = _norm2(delta)                             # cached_dist_mag, core.py:226
                pen = np.logaddexp(0, -(dist - dist_min) / k) * k            # core.py:391
                force = cfg.contact_force * delta / dist[:, None] * pen[:, None]   # core.py:392
                if a_agent and b_agent:
                    force_ratio = cfg.mass / cfg.mass            # core.py:396
                    F[:, a] = force_ratio * force + F[:, a]      # core.py:311-313
                    F[:, b] = -(1 / force_ratio) * force + F[:, b]
                elif a_agent:
                    F[:, a] = force + F[:, a]                    # core.py:401
                else:
                    F[:, b] = -force + F[:, b]                   # core.py:402 (unreachable: agents come first)
            if a_agent and W:                                    # core.py:317-327: after the pair row of a movable entity
                for w in range(W):
                    F[:, a] = F[:, a] + self._wall_force(ent[:, a], w)
        return F

    def _wall_force(self, pos: np.ndarray, w: int) -> np.ndarray:
        """core.py:407-462 (get_wall_collision_force) of one agent position [B,2] against wall w; zeros where None."""
        cfg, s = self.cfg, self.s
        horiz = s.wall_orient[:, w] == 0
        prll = np.where(horiz, pos[:, 0], pos[:, 1])             # coordinate along the wall
        perp = np.where(horiz, pos[:, 1], pos[:, 0])
        lo, hi = -s.wall_len, s.wall_len                         # wall.endpoints (:307)
        r = cfg.entity_size
        beyond = (prll < lo - r) | (prll > hi + r)               # :417-419 -> None
        partial = ~beyond & ((prll < lo) | (prll > hi))          # :420-428
        past = np.where(prll < lo, prll - lo, prll - hi)
        with np.errstate(invalid="ignore"):
            theta = np.where(partial, np.arcsin(np.where(partial, past, 0.0) / r), 0.0)
        dist_min = np.where(partial, np.cos(theta) * r + 0.5 * cfg.wall_width, r + 0.5 * cfg.wall_width)
        delta = perp - s.wall_axis[:, w]                         # :435
        dist = np.abs(delta)
        kk = cfg.wall_contact_margin
        pen = np.logaddexp(0, -(dist - dist_min) / kk) * kk      # :439
        with np.errstate(invalid="ignore", divide="ignore"):
            mag = cfg.wall_contact_force * delta / dist * pen    # :440
        f_perp = np.cos(theta) * mag                             # :444
        f_prll = np.sin(theta) * np.abs(mag)                     # :445
        fx = np.where(horiz, f_prll, f_perp)
        fy = np.where(horiz, f_perp, f_prll)
        out = np.stack([fx, fy], axis=-1)
        return np.where(beyond[:, None], 0.0, out)

    def _integrate(self, F: np.ndarray) -> None:
        """core.py:338-356 (integrate_state)."""
        cfg, s = self.cfg, self.s
        vel = s.vel * (1 - cfg.damping)
        vel = vel + (F / cfg.mass) * cfg.dt
        if cfg.max_speed is not None:
            speed = np.sqrt(np.square(vel[..., 0]) + np.square(vel[..., 1]))
            over = speed > cfg.max_speed
            with np.errstate(invalid="ignore", divide="ignore"):
                clamped = vel / speed[..., None] * cfg.max_speed
            vel = np.where(over[..., None], clamped, vel)
        s.vel = vel
        s.pos = s.pos + vel * cfg.dt
        s.p_dist = s.p_dist + _norm2(vel * cfg.dt)

    def distance_matrix(self) -> np.ndarray:
        """core.py:204-228 (calculate_distances) -> cached_dist_mag [B,E,E]."""
        ent = self._entity_pos()
        E = ent.shape[1]
        adj = np.zeros((self.B, E, E))
        for a in range(E):
            for b in range(a + 1, E):
                m = _norm2(ent[:, a] - ent[:, b])
                adj[:, a, b] = m
                adj[:, b, a] = m
        return adj

    # ------------------------------------------------------------------ scenario callbacks
    def _goal_pos(self) -> np.ndarray:
        s = self.s
        return np.take_along_axis(s.landmark_pos, s.goal_match[..., None].astype(np.int64), axis=1)

    def _fairness_param(self, i: int) -> np.ndarray:
        """navigation_graph.py:764-769 / :849-853 (+ collect_dist :914-927)."""
        s = self.s
        first = s.dists_to_goal[:, i] == -1
        mean_p = np.mean(s.p_dist, axis=1)
        std_p = np.std(s.p_dist, axis=1)
        return np.where(first, mean_p / (std_p + 0.0001),
                        s.dist_traveled_mean / (s.dist_traveled_stddev + 0.0001))

    def _collisions(self, i: int):
        """navigation_graph.py:650-661 (is_obstacle_collision, no walls), :701-705 (is_collision)."""
        cfg, s = self.cfg, self.s
        dmin = collision_dist_min(cfg)
        n_agent = np.zeros(self.B)
        for j in range(cfg.num_agents):
            if j == i:
                continue
            n_agent += _norm2(s.pos[:, j] - s.pos[:, i]) < dmin
        obst = np.zeros(self.B, dtype=bool)
        for kk in range(cfg.num_obstacles):
            obst |= _norm2(s.obstacle_pos[:, kk] - s.pos[:, i]) < dmin
        if cfg.num_walls:
            obst |= self._in_wall_box(s.pos[:, i], cfg.entity_size)
        return n_agent, obst

    def _in_wall_box(self, pos: np.ndarray, entity_size: float, sel=None) -> np.ndarray:
        """navigation_graph.py:670-683: inside the 1.05-scaled box of any wall (note the scaling of the bounds
        themselves, not of the distances, and entity_size / 2)."""
        s = self.s
        axis = s.wall_axis if sel is None else s.wall_axis[sel]
        orient = s.wall_orient if sel is None else s.wall_orient[sel]
        wl = s.wall_len if sel is None else s.wall_len[sel]
        hit = np.zeros(pos.shape[0], dtype=bool)
        h = entity_size / 2
        for w in range(self.cfg.num_walls):
            horiz = orient[:, w] == 0
            perp = np.where(horiz, pos[:, 1], pos[:, 0])
            prll = np.where(horiz, pos[:, 0], pos[:, 1])
            hit |= ((1.05 * (axis[:, w] - h) <= perp) & (perp <= 1.05 * (axis[:, w] + h)) &
                    (1.05 * (-wl - h) <= prll) & (prll <= 1.05 * (wl + h)))
        return hit

    def _observation(self, i: int, goal: np.ndarray) -> np.ndarray:
        """navigation_graph.py:826-857: [vel, pos, goal - pos, fairness_param]."""
        s = self.s
        return np.concatenate([s.vel[:, i], s.pos[:, i], goal[:, i] - s.pos[:, i],
                               self._fairness_param(i)[:, None]], axis=1)

    def _reward(self, i: int, goal: np.ndarray) -> np.ndarray:
        """navigation_graph.py:760-824."""
        cfg, s = self.cfg, self.s
        d = _norm2(s.pos[:, i] - goal[:, i])
        rew = np.where(d < cfg.min_dist_thresh, cfg.goal_rew, -d)             # :779-782
        n_agent, obst = self._collisions(i)
        rew = rew - cfg.collision_rew * n_agent                                 # :784-790
        rew = rew - cfg.collision_rew * obst                                    # :792-794
        if cfg.fairness_reward:
            fair = cfg.fair_rew * np.tanh(self._fairness_param(i) - cfg.zeroshift)   # :806-808
            fair = np.where(fair < -2, -2.0, fair)                              # :809-810
            rew = rew + fair
        return np.clip(rew, -2 * cfg.collision_rew, cfg.goal_rew + cfg.fair_rew)     # :824

    def _info(self, i: int, goal: np.ndarray) -> None:
        """navigation_graph.py:577-647 (stateful part)."""
        cfg, s = self.cfg, self.s
        d = _norm2(s.pos[:, i] - goal[:, i])
        latch = (d < cfg.min_dist_thresh) & (s.times_required[:, i] == -1)        # :587
        s.times_required[:, i] = np.where(latch, s.step * cfg.dt, s.times_required[:, i])
        s.dists_to_goal[:, i] = np.where(latch, s.p_dist[:, i], s.dists_to_goal[:, i])
        s.dist_left_to_goal[:, i] = np.where(latch, d, s.dist_left_to_goal[:, i])
        open_ = s.times_required[:, i] == -1                                      # :595
        s.dists_to_goal[:, i] = np.where(open_, s.p_dist[:, i], s.dists_to_goal[:, i])
        s.dist_left_to_goal[:, i] = np.where(open_, d, s.dist_left_to_goal[:, i])
        n_agent, obst = self._collisions(i)
        s.num_obstacle_collisions[:, i] += obst                                   # :602-603
        s.num_agent_collisions[:, i] += n_agent                                   # :604-613
        s.dist_traveled_mean = np.mean(s.dists_to_goal, axis=1)                   # :617
        s.dist_traveled_stddev = np.std(s.dists_to_goal, axis=1)                  # :618

    def _node_obs(self, goal: np.ndarray) -> np.ndarray:
        """navigation_graph.py:941-1035 + :1079-1124 (relative features) -> [B,N,E,11];
        :1058-1077 (global features [vel, pos, goal, type], the same rows for every agent) -> [B,N,E,7]."""
        cfg, s = self.cfg, self.s
        N, O, E = cfg.num_agents, cfg.num_obstacles, cfg.num_entities
        W = cfg.num_walls
        ent_pos = self._entity_pos()
        ent_vel = np.concatenate([s.vel, np.zeros((self.B, N + O + W, 2))], axis=1)
        if cfg.graph_feat_type == "global":
            if W:
                raise ValueError("wall entities are not supported by the global features (navigation_graph.py:1074-1075)")
            g = ent_pos.copy()
            g[:, :N] = goal
            typ = np.concatenate([np.zeros(N), np.ones(N), 2.0 * np.ones(O)])
            rows = np.concatenate([ent_vel, ent_pos, g, np.broadcast_to(typ[None, :, None], (self.B, E, 1))], axis=2)
            return np.broadcast_to(rows[:, None], (self.B, N, E, 7)).copy()
        out = np.zeros((self.B, N, E, 11))
        for a in range(N):
            rel_pos = ent_pos - s.pos[:, a:a + 1]
            rel_vel = ent_vel - s.vel[:, a:a + 1]
            rel_goal = rel_pos.copy()
            rel_goal[:, :N] = goal - s.pos[:, a:a + 1]
            out[:, a, :, 0:2] = rel_vel
            out[:, a, :, 2:4] = rel_pos
            out[:, a, :, 4:6] = rel_goal
            out[:, a, :, 6:8] = rel_pos
            out[:, a, :, 8:10] = rel_pos
            out[:, a, :N, 10] = 0.0          # entity_mapping (navigation_graph.py:22)
            out[:, a, N:2 * N, 10] = 1.0
            out[:, a, 2 * N:2 * N + O, 10] = 2.0
            for w in range(W):               # :1108-1118: corner offsets instead of the repeated rel_pos
                e = 2 * N + O + w            # (endpoints[0], axis + width/2) and (endpoints[1], axis - width/2) as
                o_c = np.stack([-s.wall_len, s.wall_axis[:, w] + cfg.wall_width / 2], axis=-1)   # (x, y), whatever the orientation
                d_c = np.stack([s.wall_len, s.wall_axis[:, w] - cfg.wall_width / 2], axis=-1)
                out[:, a, e, 6:8] = o_c - s.pos[:, a]
                out[:, a, e, 8:10] = d_c - s.pos[:, a]
                out[:, a, e, 10] = 3.0
        return out

    # ------------------------------------------------------------------ env step
    def step(self, actions=None, onehot=None, autoreset: bool = True) -> Dict[str, np.ndarray]:
        """environment.py:816-877 (MultiAgentGraphEnv.step) + env_wrappers.py:856-865 (auto-reset).

        Returns dict with obs [B,N,7], node_obs [B,N,E,11], adj [B,E,E], reward [B,N],
        done [B,N] bool, info {key: [B,N]} (terminal values on auto-reset steps), reset [B] bool.
        """
        cfg, s = self.cfg, self.s
        N = cfg.num_agents
        s.step = s.step + 1                                           # environment.py:819, :823
        u = self._action_u(actions, onehot)
        F = self._forces(u)                                           # world.step(), core.py:250-274
        self._integrate(F)
        adj = self.distance_matrix()
        goal = self._goal_pos()
        obs = np.zeros((self.B, N, 7))
        rew = np.zeros((self.B, N))
        info = {k: np.zeros((self.B, N)) for k in INFO_KEYS}
        # time accumulates by repeated `+= dt` (core.py:355); same for every agent
        t_acc = np.zeros(self.B)
        for kk in range(int(s.step.max()) if self.B else 0):
            t_acc = np.where(kk < s.step, t_acc + cfg.dt, t_acc)
        for i in range(N):                                            # environment.py:832-864
            obs[:, i] = self._observation(i, goal)
            rew[:, i] = self._reward(i, goal)
            self._info(i, goal)
            tm = np.mean(s.times_required, axis=1)                    # navigation_graph.py:620-621
            ts = np.std(s.times_required, axis=1)
            info["individual_reward"][:, i] = rew[:, i]
            info["Dist_to_goal"][:, i] = s.dist_left_to_goal[:, i]
            info["Time_req_to_goal"][:, i] = s.times_required[:, i]
            info["Num_agent_collisions"][:, i] = s.num_agent_collisions[:, i]
            info["Num_obst_collisions"][:, i] = s.num_obstacle_collisions[:, i]
            info["Distance_mean"][:, i] = s.dist_traveled_mean
            info["Distance_variance"][:, i] = s.dist_traveled_stddev
            info["Mean_by_variance"][:, i] = s.dist_traveled_mean / (s.dist_traveled_stddev + 0.0001)
            info["Dists_traveled"][:, i] = s.dists_to_goal[:, i]
            info["Time_taken"][:, i] = t_acc
            info["Time_mean"][:, i] = tm
            info["Time_stddev"][:, i] = ts
            info["Time_mean_by_stddev"][:, i] = tm / (ts + 0.0001)
            info["Min_time_to_goal"][:, i] = s.min_time[:, i]
        node_obs = self._node_obs(goal)
        done_env = s.step >= cfg.episode_length                       # environment.py:237-247
        done = np.repeat(done_env[:, None], N, axis=1)
        if cfg.collaborative:                                         # environment.py:867-870
            rew = np.repeat(rew.sum(axis=1, keepdims=True), N, axis=1)
        reset = np.zeros(self.B, dtype=bool)
        if autoreset and done_env.any():                              # env_wrappers.py:859-865
            reset = done_env.copy()
            r = self.reset(mask=reset)
            obs = np.where(reset[:, None, None], r["obs"], obs)
            node_obs = np.where(reset[:, None, None, None], r["node_obs"], node_obs)
            adj = np.where(reset[:, None, None], r["adj"], adj)
        self.last_info = info
        return dict(obs=obs, node_obs=node_obs, adj=adj, reward=rew, done=done, info=info, reset=reset)

    def observe(self) -> Dict[str, np.ndarray]:
        """environment.py:882-898: obs / node_obs / adj of the current state (no state change)."""
        goal = self._goal_pos()
        N = self.cfg.num_agents
        obs = np.stack([self._observation(i, goal) for i in range(N)], axis=1)
        return dict(obs=obs, node_obs=self._node_obs(goal), adj=self.distance_matrix())

    # ------------------------------------------------------------------ reset
    def _draw(self, envs: np.ndarray, draw_idx: np.ndarray):
        """One 2-D uniform draw per env: Philox counter (draw, episode, env_lo, env_hi), key = seed.
        Returns float32 (ux, uy) in [0,1) with 24 bits."""
        g = (envs + self.env_offset).astype(np.uint64)
        r0, r1, _, _ = philox4x32_10(
            draw_idx.astype(np.uint32), self.s.episode[envs].astype(np.uint32),
            (g & np.uint64(0xFFFFFFFF)).astype(np.uint32), (g >> np.uint64(32)).astype(np.uint32),
            np.uint32(self.seed & 0xFFFFFFFF), np.uint32((self.seed >> 32) & 0xFFFFFFFF))
        return u01_24(r0), u01_24(r1)

    MAX_DRAWS = 4096

    def reset(self, mask: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
        """navigation_graph.py:212-262 (reset_world) + :264-570 (random_scenario), with the device's
        Philox stream instead of numpy's global MT19937 (acceptance rules identical):

        * obstacles ``0.8 * U(-ws/2, ws/2)^2`` (:271-275)
        * agents  ``U(-ws/2, ws/2)^2``, rejected while closer than 1.05*(r+r) to an obstacle
          (:650-661) or an already placed agent (:686-698)   (:389-456)
        * goals   ``0.8 * U(...)``, rejected vs obstacles and already placed goals (:472-535, :707-716)
        * ``min_time`` with the PREVIOUS goal_match_index (:545-547, :719-728)
        * lexifair assignment on cdist(agent_pos, goal_pos) (:555-561)
        Positions are float32 values (the device state dtype); predicates are float64.
        """
        cfg, s = self.cfg, self.s
        N, O = cfg.num_agents, cfg.num_obstacles
        if mask is None:
            mask = np.ones(self.B, dtype=bool)
        envs = np.nonzero(mask)[0]
        nb = envs.size
        if nb:
            ws = np.float32(cfg.world_size)
            half = np.float32(cfg.world_size / 2)
            dmin = collision_dist_min(cfg)
            draw = np.zeros(nb, dtype=np.int64)

            def uniform(sel):
                ux, uy = self._draw(envs[sel], draw[sel])
                draw[sel] += 1
                return np.stack([ws * ux - half, ws * uy - half], axis=-1).astype(np.float32)

            all_sel = np.arange(nb)
            ob = np.zeros((nb, O, 2), dtype=np.float32)
            for kk in range(O):
                ob[:, kk] = np.float32(0.8) * uniform(all_sel)
            W = cfg.num_walls
            if W:                                                      # :287-324, after the obstacles
                ux, _ = self._draw(envs, draw); draw += 1
                wp = (np.float32(0.2) + np.float32(0.7) * ux) * np.float32(cfg.world_size / 2)    # U(0.2, 0.9) * ws / 2
                axis = np.stack([wp, -wp], axis=-1)[:, :W]
                orient = np.zeros((nb, W), dtype=np.int64)
                for w in range(W):
                    uo, _ = self._draw(envs, draw); draw += 1
                    orient[:, w] = (uo >= np.float32(0.5)).astype(np.int64)     # np.random.choice(['H', 'V'])
                s.wall_axis[envs] = axis.astype(np.float64)
                s.wall_orient[envs] = orient
            ag = np.zeros((nb, N, 2), dtype=np.float32)
            lm = np.zeros((nb, N, 2), dtype=np.float32)

            def place(dst, shrink, others_fn):
                for i in range(N):
                    pending = all_sel.copy()
                    while pending.size:
                        cand = uniform(pending)
                        if shrink:
                            cand = np.float32(0.8) * cand
                        c64 = cand.astype(np.float64)
                        bad = np.zeros(pending.size, dtype=bool)
                        for kk in range(O):
                            bad |= _norm2(ob[pending, kk].astype(np.float64) - c64) < dmin
                        for j in range(i):
                            bad |= _norm2(dst[pending, j].astype(np.float64) - c64) < dmin
                        if W:                                          # is_obstacle_collision's wall boxes (:670-683)
                            bad |= self._in_wall_box(c64, cfg.entity_size, sel=envs[pending])
                        bad &= draw[pending] < self.MAX_DRAWS          # give up rejecting (device cap)
                        ok = ~bad
                        dst[pending[ok], i] = cand[ok]
                        pending = pending[bad]

            place(ag, False, None)
            place(lm, True, None)
            s.obstacle_pos[envs] = ob
            s.pos[envs] = ag
            s.landmark_pos[envs] = lm
            s.vel[envs] = 0.0
            s.p_dist[envs] = 0.0                                       # :239
            s.step[envs] = 0                                           # :215, environment.py:883
            s.times_required[envs] = -1.0                              # :217-218
            s.dists_to_goal[envs] = -1.0
            s.dist_left_to_goal[envs] = -1.0                           # :221
            s.num_obstacle_collisions[envs] = 0.0                      # :223-225
            s.num_agent_collisions[envs] = 0.0
            ag64, lm64 = ag.astype(np.float64), lm.astype(np.float64)
            if cfg.max_speed is not None:                              # :545-547
                old_goal = np.take_along_axis(lm64, s.goal_match[envs][..., None], axis=1)
                s.min_time[envs] = _norm2(ag64 - old_goal) / cfg.max_speed
            costs = _norm2(ag64[:, :, None, :] - lm64[:, None, :, :])  # cdist, :555
            s.goal_match[envs] = _lexifair.lexifair(costs)             # :556-558
            s.episode[envs] += 1
        out = self.observe()
        return out
