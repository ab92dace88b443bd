"""Drop-in mirror of the reference's `AssemblySwarmEnv` / `AssemblySwarmWrapper` on top of the GPU simulator.

Same class names, method names, argument meaning, return shapes/dtypes and attribute surface as
cus_gym/gym/envs/customized_envs/assembly.py (ENV) and cus_gym/gym/wrappers/customized_envs/assembly_wrapper.py (WRAP),
so that marl_llm/train/train_assembly.py and eval/eval_assembly.py see the env they expect (SURVEY.md §8b):

    env = AssemblySwarmWrapper(AssemblySwarmEnv(), args)
    obs = env.reset()                                   # (192, n_a) float64                     ENV:156-223
    obs, rew, done, info, a_prior = env.step(a)         # a: (2, n_a) float32/64                  ENV:487-666
    env.p, env.dp, env.env.grid_center = ...            # readable and writable (eval_assembly.py:34-57,137-151)

`num_envs > 1` gives a vectorised variant with a leading batch axis on every array (not in the reference).
All arithmetic runs in the sm_100a kernels (marl_llm_b200/csrc); there is no CPU fallback.  render("rgb_array") returns frames
drawn on the device (marl_llm_b200/render.py); render() in "human" mode draws nothing and returns None.
"""
import pickle

import numpy as np
import torch

from .batched import BatchedAssemblySim
from .render import SwarmRenderer

RGB_ARRAY_SIZE = 480        # render("rgb_array") frames are RGB_ARRAY_SIZE x RGB_ARRAY_SIZE pixels of the arena


class Box:
    """The one gym.spaces member the scripts touch (ENV:802,806): shape / dtype / low / high."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), dtype

    def sample(self):
        return np.random.uniform(-1, 1, self.shape).astype(self.dtype)


class AssemblySwarmEnv:
    metadata = {"render.modes": ["human", "rgb_array"], "video.frames_per_second": 45}

    def __init__(self, num_envs=1, device=0):
        # constants of ENV:18-90 that callers may read
        self.num_envs, self.device = int(num_envs), device
        self.reward_sharing_mode = "individual"
        self.penalize_entering = self.penalize_interaction = self.penalize_exploration = True
        self.dim, self.n_a, self.n_o = 2, 10, 0
        self.topo_nei_max = 6
        self.act_dim_agent = self.dim
        self.m_a, self.size_a = 1, 0.035
        self.d_sen, self.r_avoid = 3, 0.15
        self.Vel_max, self.Vel_min, self.Acc_max = 0.8, 0.0, 1
        self.boundary_width_half = self.boundary_height_half = 2.4
        self.bound_center = np.zeros(2)
        self.k_ball, self.k_wall, self.c_wall = 30, 100, 5
        self.simulation_time, self.dt, self.n_frames, self.sensitivity = 0, 0.1, 1, 1
        self._sim = None
        self._rend = None
        self.render_traj, self.traj_len = False, 15
        self._grid_dirty = False
        self.unwrapped = self

    # ---------------------------------------------------------------------------------------- ENV:92-154
    def __reinit__(self, args):
        self.n_a = args.n_a
        self.render_traj, self.traj_len = getattr(args, "render_traj", False), getattr(args, "traj_len", 15)
        self.is_collected, self.video = getattr(args, "is_collected", False), getattr(args, "video", False)
        self.is_boundary = args.is_boundary
        self.is_periodic = not self.is_boundary
        self.dynamics_mode, self.agent_strategy = args.dynamics_mode, args.agent_strategy
        self.is_con_self_state, self.is_feature_norm = args.is_con_self_state, args.is_feature_norm
        self.training_method = args.training_method
        self.alpha = 1
        if self.dynamics_mode != "Cartesian":
            raise NotImplementedError("only dynamics_mode='Cartesian' exists in the reference (ENV:141-146)")
        if self.agent_strategy not in ("input", "random", "rule", "llm"):
            raise ValueError("Wrong in Step function")                   # ENV:602-603
        if self.agent_strategy in ("rule", "llm") and self.is_periodic:
            raise NotImplementedError("the 'rule' / 'llm' strategies are implemented for is_boundary=True")
        self.results_file = args.results_file
        if isinstance(self.results_file, dict):
            loaded = self.results_file
        else:
            with open(self.results_file, "rb") as f:
                loaded = pickle.load(f)
        self.l_cells = loaded["l_cell"]
        self.grid_center_origins = loaded["grid_coords"]
        self.binary_images = loaded.get("binary_image", [None] * len(self.l_cells))
        self.shape_bound_points_origins = loaded["shape_bound_points"]
        self.num_train_shape = len(self.l_cells)
        self.n_gs = [g.shape[0] for g in self.grid_center_origins]
        self.r_avoid = round(np.sqrt(4 * np.min(self.n_gs) / (self.n_a * np.pi)) * np.min(self.l_cells), 2)   # ENV:124
        self.num_obs_grid_max, self.num_occupied_grid_max = 80, 200
        self_flag = 1 if self.is_con_self_state else 0
        self.obs_dim_agent = 2 * self.dim * (self.topo_nei_max + 1 + self_flag) + self.dim * self.num_obs_grid_max   # ENV:801
        self.observation_space = Box(-np.inf, np.inf, (self.obs_dim_agent, self.n_a), np.float32)
        self.action_space = Box(-np.inf, np.inf, (self.act_dim_agent, self.n_a), np.float32)
        self.m = np.array([self.m_a] * self.n_a)
        self.size = np.array([self.size_a] * self.n_a)
        np.random.choice([True, False], size=(self.n_a, self.n_a))      # ENV:133 consumes NumPy-global RNG state
        self.shape_frequency = np.zeros_like(self.l_cells)
        self.d_sen = 0.4                                                # ENV:199 (set at reset in the reference)
        self._n_g_cap = max(int(max(self.n_gs)), 1)
        self._make_sim(self._n_g_cap)

    def _make_sim(self, n_g_cap):
        if self._sim is not None:
            self._sim.close()
        self._n_g_cap = n_g_cap
        self._sim = BatchedAssemblySim(
            self.num_envs, self.n_a, n_g_cap, self.r_avoid, device=self.device, out_dtype=torch.float64,
            emit_indices=True, want_prior=(self.training_method == "llm_rl"), is_con_self_state=self.is_con_self_state,
            is_periodic=self.is_periodic, d_sen=self.d_sen, size_a=self.size_a, k_ball=float(self.k_ball),
            k_wall=float(self.k_wall), c_wall=float(self.c_wall), dt=self.dt, vel_max=self.Vel_max, mass=float(self.m_a),
            half_width=self.boundary_width_half, half_height=self.boundary_height_half)
        # the shape library (ENV:116-119): grids installed by reset() / by the caller are recognised as rigid transforms of
        # these shapes, which lets the simulator use its lookup-scan kernel (results are identical without it)
        if n_g_cap >= max(self.n_gs):
            self._sim.set_shapes([np.ascontiguousarray(np.asarray(g, dtype=np.float64).T) for g in self.grid_center_origins],
                                 [float(v) for v in self.l_cells])

    # ---------------------------------------------------------------------------------------- helpers
    def _squeeze(self, a):
        return a[0] if self.num_envs == 1 else a

    def _host(self, t):
        return self._squeeze(t.cpu().numpy())

    def _push_grid(self):
        E = self.num_envs
        poses = getattr(self, "_poses", None)
        if poses is not None and self._sim.shapes_installed:
            # reset() chose (shape, angle, offset) itself and NumPy's grid equals the device's own R.origin + off bit for bit
            # (checked in _reset_one): hand over the pose, the device rebuilds the identical grid and knows the pose exactly
            k, c, s, ox, oy = (np.array(v) for v in zip(*poses))
            self._sim.set_grid_pose(k, c, s, ox, oy)
            self._grid_dirty = False
            return
        grids = [self._grid_center] if E == 1 else list(self._grid_center)
        n_g = max(g.shape[1] for g in grids)
        if n_g > self._n_g_cap:                                          # eval may install a bigger shape
            # The handle is rebuilt with a larger cell capacity.  Everything the next step() reads from the last observation
            # moves over (eval_assembly.py:34-57 swaps the shape mid-episode, with no reset): p / dp, the neighbour list the
            # prior is computed from (ENV:613-624), in_flags, the outputs; the new handle is then marked as observed.
            old = self._sim
            keep = {k: getattr(old, k).clone() for k in ("p", "dp", "neighbor_index", "in_flags", "nearest_cell", "obs", "reward",
                                                         "sensed_index", "occupied_index")}
            observed = old.observed
            self._make_sim(n_g)
            for k, v in keep.items():
                getattr(self._sim, k).copy_(v)
            if observed:
                self._sim.restore_observation()
            self._sim.mark_state_dirty()
        blocks, ng = self._sim.pack_grids(grids, self._n_g_cap)
        l_cell = np.broadcast_to(np.asarray(self._l_cell, dtype=np.float64), (E,))
        self._sim.set_grid(blocks, ng, l_cell)
        self._grid_dirty = False

    # state the callers read and overwrite (eval_assembly.py:34-57, 137-151)
    @property
    def p(self):
        return self._host(self._sim.p)

    @p.setter
    def p(self, v):
        self._sim.p.copy_(torch.as_tensor(np.asarray(v, dtype=np.float64)).reshape(self._sim.p.shape))
        self._sim.mark_state_dirty()

    @property
    def dp(self):
        return self._host(self._sim.dp)

    @dp.setter
    def dp(self, v):
        self._sim.dp.copy_(torch.as_tensor(np.asarray(v, dtype=np.float64)).reshape(self._sim.dp.shape))
        self._sim.mark_state_dirty()

    @property
    def grid_center(self):
        return self._grid_center

    @grid_center.setter
    def grid_center(self, v):
        self._grid_center = np.ascontiguousarray(v, dtype=np.float64) if self.num_envs == 1 else v
        self._grid_dirty = True
        self._poses = None             # a caller-provided grid: the simulator recognises its pose itself (or uses the general scan)

    @property
    def l_cell(self):
        return self._l_cell

    @l_cell.setter
    def l_cell(self, v):
        self._l_cell = v
        self._grid_dirty = True
        self._poses = None

    @property
    def n_g(self):
        g = self._grid_center
        return g.shape[1] if self.num_envs == 1 else [x.shape[1] for x in g]

    @n_g.setter
    def n_g(self, v):      # derived from grid_center; the assignment at eval_assembly.py:44 is accepted and ignored
        pass

    obs = property(lambda self: self._host(self._sim.obs))
    neighbor_index = property(lambda self: self._host(self._sim.neighbor_index))
    in_flags = property(lambda self: self._host(self._sim.in_flags))
    sensed_index = property(lambda self: self._host(self._sim.sensed_index))
    occupied_index = property(lambda self: self._host(self._sim.occupied_index))

    # ---------------------------------------------------------------------------------------- ENV:156-223
    def _reset_one(self):
        """One env's domain randomisation with the reference's NumPy-global RNG call order."""
        k = np.random.randint(0, self.num_train_shape)
        self.shape_frequency[k] += 1
        l_cell = self.l_cells[k]
        origin = np.asarray(self.grid_center_origins[k]).T
        self.target_shape = self.binary_images[k]
        sbp_origin = np.asarray(self.shape_bound_points_origins[k])
        ang = np.pi * np.random.uniform(-1, 1)
        R = np.array([[np.cos(ang), np.sin(ang)], [-np.sin(ang), np.cos(ang)]])
        origin = np.dot(R, origin)
        np.random.uniform(-1.2, 1.2, (2, 1))                            # ENV:182, drawn and overwritten
        hw, hh = self.boundary_width_half, self.boundary_height_half
        off = np.array([[np.random.uniform(-hw + 1, hw - 1), np.random.uniform(-hh + 1, hh - 1)]]).T
        grid = origin.copy() + off
        sbp = np.hstack((sbp_origin[:2] + off[0, 0], sbp_origin[2:] + off[1, 0]))
        if np.random.uniform(-1, 1) > 0:
            p = np.concatenate((np.random.uniform(-hw, hw, (1, self.n_a)), np.random.uniform(-hh, hh, (1, self.n_a))), axis=0)
        else:
            p = np.random.uniform(-1, 1, (2, self.n_a)) + np.array(
                [[np.random.uniform(-hw + 1, hw - 1), np.random.uniform(-hh + 1, hh - 1)]]).T
        dp = np.random.uniform(-0.5, 0.5, (self.dim, self.n_a))
        # does NumPy's np.dot(R, origin) + off equal the separately rounded R.origin + off the device computes?  (it does unless
        # the BLAS behind np.dot contracts into FMAs); if so the pose can be handed over instead of the grid
        o0 = np.asarray(self.grid_center_origins[k], dtype=np.float64).T
        alt = BatchedAssemblySim.grid_from_pose(o0, R[0, 0], R[0, 1], off[0, 0], off[1, 0])
        self._pose_one = (k, R[0, 0], R[0, 1], off[0, 0], off[1, 0]) if np.array_equal(alt, grid) else None
        return l_cell, origin, grid, sbp_origin, sbp, p, dp

    def reset(self):
        self.simulation_time = 0
        outs, poses = [], []
        for _ in range(self.num_envs):
            outs.append(self._reset_one())
            poses.append(self._pose_one)
        one = self.num_envs == 1
        self._l_cell = outs[0][0] if one else np.array([o[0] for o in outs])
        self.grid_center_origin = outs[0][1] if one else [o[1] for o in outs]
        self._grid_center = outs[0][2] if one else [o[2] for o in outs]
        self.shape_bound_points_origin = outs[0][3] if one else [o[3] for o in outs]
        self.shape_bound_points = outs[0][4] if one else [o[4] for o in outs]
        self.boundary_pos = np.array([-self.boundary_width_half, self.boundary_height_half,
                                      self.boundary_width_half, -self.boundary_height_half], dtype=np.float64)
        self.d_sen = 0.4
        self._poses = poses if all(q is not None for q in poses) else None
        self._push_grid()
        self._sim.set_state(np.stack([o[5] for o in outs]), np.stack([o[6] for o in outs]))
        self.ddp = np.zeros((2, self.n_a))
        self.heading = np.zeros((self.dim, self.n_a))
        self._sim.observe()
        if self.render_traj:
            self._renderer().clear()
            self._renderer().record()
        return self.obs

    # ---------------------------------------------------------------------------------------- ENV:487-666
    def step(self, a):
        self.simulation_time += self.dt
        if self._grid_dirty:
            self._push_grid()
        # ENV:519-601: 'input' uses the caller's action; 'random' draws it from NumPy's global stream like the reference;
        # 'rule' / 'llm' are evaluated on the device from the pre-step state (swarm_strategy_actions)
        if self.agent_strategy == "random":
            a = np.random.uniform(-1, 1, (self.num_envs, 2, self.n_a) if self.num_envs > 1 else (2, self.n_a))   # ENV:522-523
        if self.agent_strategy in ("rule", "llm"):
            act = self._sim.strategy_actions(self.agent_strategy)
            a = act.cpu().numpy().reshape((self.num_envs, 2, self.n_a) if self.num_envs > 1 else (2, self.n_a))
        else:
            a = np.ascontiguousarray(a)
            if a.dtype not in (np.float32, np.float64):
                a = a.astype(np.float64)
            act = torch.from_numpy(a).reshape(self.num_envs, 2, self.n_a).to(self._sim.device)
        obs, rew, done, _, prior = self._sim.step(act)
        if self.render_traj:
            self._renderer().record()
        info = np.array([None, None, None]).reshape(3, 1)               # ENV:484-485
        u = a.astype(np.float64)
        last = u if self.is_collected else (self._host(prior) if prior is not None else None)   # ENV:663-666
        return self._host(obs), self._host(rew), self._host(done), info, last

    def _renderer(self):
        """The renderer of every env of the current handle (rebuilt with the handle, keeping the recorded trail)."""
        r = self._rend
        if r is None or r.sim is not self._sim:
            new = SwarmRenderer(self._sim, np.arange(self.num_envs), RGB_ARRAY_SIZE, RGB_ARRAY_SIZE,
                                trail_len=self.traj_len if self.render_traj else 0)
            if r is not None and r.trail is not None and new.trail is not None:
                new.trail.copy_(r.trail)
                new.trail_len, new.trail_head = r.trail_len, r.trail_head
            self._rend = r = new
        return r

    def render(self, mode="human"):
        """ENV:668-747 draws the swarm with matplotlib.  mode="rgb_array": a uint8 [480, 480, 3] frame of the arena drawn on the
        device ([E, 480, 480, 3] with num_envs > 1): the env's target cells, the trails of the last traj_len positions when
        render_traj is set, and the agents, green inside the shape and red outside (DESIGN.md §10).  This draws the env's actual,
        rotated cells, where the reference shows the un-rotated source bitmap at shape_bound_points.  Any other mode draws
        nothing and returns None, which keeps train_assembly.py:93-94 and eval_assembly.py:147 unchanged."""
        if mode != "rgb_array":
            return None
        if self._grid_dirty:
            self._push_grid()
        return self._host(self._renderer().render())

    def close(self):
        if self._sim is not None:
            self._sim.close()
            self._sim = None
        self._rend = None


class Agent:
    def __init__(self, adversary=False):
        self.adversary = adversary


class AssemblySwarmWrapper:
    """WRAP:18-129: re-inits the env with `args`, exposes num_agents/agents/agent_types and the three eval metrics
    (computed on the device by `k_metrics`; they are not on the step path)."""

    def __init__(self, env, args):
        self.env = env
        env.__reinit__(args)
        self.num_agents = env.n_a
        self.agents = [Agent() for _ in range(self.num_agents)]
        self.agent_types = ["agent"]
        self.action_space, self.observation_space = env.action_space, env.observation_space

    def __getattr__(self, name):                       # gym.Wrapper.__getattr__ (core.py:225-229)
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.env, name)

    @property
    def unwrapped(self):
        return self.env

    def reset(self, **kw):
        return self.env.reset(**kw)

    def step(self, action):
        return self.env.step(action)

    def render(self, mode="human", **kw):
        return self.env.render(mode, **kw)

    def close(self):
        return self.env.close()

    def _metric(self, k):
        env = self.env
        if env._grid_dirty:
            env._push_grid()
        m = env._sim.metrics()[:, k].cpu().numpy()
        return float(m[0]) if env.num_envs == 1 else m

    def coverage_rate(self):                           # WRAP:48-72, on the device (swarm_metrics)
        return self._metric(0)

    def distribution_uniformity(self):                 # WRAP:74-101
        return self._metric(1)

    def voronoi_based_uniformity(self):                # WRAP:103-129
        return self._metric(2)
