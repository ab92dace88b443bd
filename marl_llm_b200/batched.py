"""Device-resident batch of assembly environments stepped by the fused sm_100a kernel.

Host side of the batched C ABI (include/swarm_b200.h, group 2).  torch is used for what the task statement
says it is for: device memory (the state / output tensors below are plain torch tensors whose data_ptr()s are
handed to the library once) and streams.  All arithmetic happens in marl_llm_b200/csrc.

Per-env layouts equal the reference's (cus_gym/gym/envs/customized_envs/assembly.py):
    p, dp            [E, 2, n_a]        float64      assembly.py:203-215
    obs              [E, obs_dim, n_a]  out dtype    assembly.py:227,  AssemblyEnv.cpp:324-328
    reward           [E, 1, n_a]        out dtype    assembly.py:353
    done             [E, 1, n_a]        bool, always False (assembly.py:480-482)
    a_prior          [E, 2, n_a]        out dtype    assembly.py:612
    neighbor_index   [E, n_a, 6]  in_flags [E, n_a]  sensed_index [E, n_a, 80]  occupied_index [E, n_a, 200]  int32
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import SwarmBuffers, SwarmConfig, SwarmError, check

TOPO_NEI_MAX = 6          # assembly.py:34
NUM_OBS_GRID_MAX = 80     # assembly.py:128
NUM_OCC_GRID_MAX = 200    # assembly.py:130


def r_avoid_for(n_a, n_gs, l_cells):
    """assembly.py:124"""
    return round(float(np.sqrt(4 * np.min(n_gs) / (n_a * np.pi)) * np.min(l_cells)), 2)


class BatchedAssemblySim:
    """E assembly envs on one device.  To save env states and load them back into this or another handle of the same
    configuration (several policies from the same start states, branching rollouts, one env cloned into others), use
    marl_llm_b200.state_store.StateStore rather than copying the buffers by hand."""

    def __init__(self, num_envs, n_a, n_g_max, r_avoid, *, device=0, out_dtype=torch.float32, emit_indices=False,
                 want_prior=True, is_con_self_state=True, is_periodic=False, d_sen=0.4, size_a=0.035, k_ball=30.0,
                 k_wall=100.0, c_wall=5.0, dt=0.1, vel_max=0.8, mass=1.0, half_width=2.4, half_height=2.4,
                 exact_occupancy=False, brute_force_scan=False, exact_reward_sums=False, obs_layout="reference", guard_bytes=0):
        if not torch.cuda.is_available():
            raise SwarmError("BatchedAssemblySim needs a CUDA device; there is no CPU fallback")
        if out_dtype not in (torch.float32, torch.float64):
            raise ValueError("out_dtype must be torch.float32 or torch.float64")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.E, self.n_a, self.n_g_max = int(num_envs), int(n_a), int(n_g_max)
        self.out_dtype = out_dtype
        self.emit_indices = bool(emit_indices)
        self.want_prior = bool(want_prior)
        self.r_avoid, self.d_sen = float(r_avoid), float(d_sen)

        cfg = SwarmConfig()
        cfg.struct_size = C.sizeof(SwarmConfig)
        cfg.device = self.device.index
        cfg.num_envs, cfg.n_a, cfg.n_g_max = self.E, self.n_a, self.n_g_max
        cfg.topo_nei_max, cfg.num_obs_grid_max, cfg.num_occupied_grid_max = TOPO_NEI_MAX, NUM_OBS_GRID_MAX, NUM_OCC_GRID_MAX
        cfg.is_con_self_state, cfg.is_periodic, cfg.want_prior = int(is_con_self_state), int(is_periodic), int(want_prior)
        cfg.out_dtype = _lib.SWARM_F32 if out_dtype == torch.float32 else _lib.SWARM_F64
        cfg.emit_indices, cfg.exact_occupancy = int(emit_indices), int(exact_occupancy)
        cfg.brute_force_scan = int(brute_force_scan)
        cfg.debug_flags = 1 if exact_reward_sums else 0
        cfg.obs_layout = {"reference": _lib.SWARM_OBS_REFERENCE, "agent_major": _lib.SWARM_OBS_AGENT_MAJOR}[obs_layout]
        self.obs_layout = obs_layout
        cfg.d_sen, cfg.r_avoid, cfg.size_a = d_sen, r_avoid, size_a
        cfg.k_ball, cfg.k_wall, cfg.c_wall = k_ball, k_wall, c_wall
        cfg.dt, cfg.vel_max, cfg.mass = dt, vel_max, mass
        cfg.boundary_pos[:] = [-half_width, half_height, half_width, -half_height]      # assembly.py:193-196
        self.cfg = cfg
        self.obs_dim = int(self.lib.swarm_obs_dim(C.byref(cfg)))
        self.n_g_pad = int(self.lib.swarm_grid_pad(self.n_g_max))

        E, n, dev = self.E, self.n_a, self.device
        # guard_bytes > 0 (tests): every device buffer sits between two guard zones filled with 0xA5; check_guards() verifies
        # that no kernel wrote outside its arrays (compute-sanitizer is not available on the GPU pool)
        self._guards = []
        gb = (int(guard_bytes) + 255) // 256 * 256

        def z(*shape, dtype):
            if not gb:
                return torch.zeros(*shape, dtype=dtype, device=dev)
            numel = int(np.prod(shape)) if shape else 1
            nbytes = (numel * torch.empty((), dtype=dtype).element_size() + 255) // 256 * 256
            raw = torch.full((gb + nbytes + gb,), 0xA5, dtype=torch.uint8, device=dev)
            raw[gb:gb + nbytes] = 0
            self._guards.append((raw, gb, nbytes))
            return raw[gb:gb + numel * torch.empty((), dtype=dtype).element_size()].view(dtype).view(*shape)
        self.p = z(E, 2, n, dtype=torch.float64)
        self.dp = z(E, 2, n, dtype=torch.float64)
        self._grid = z(E, self.n_g_pad, 2, dtype=torch.float64)
        self._n_g = z(E, dtype=torch.int32)
        self._in_thresh = z(E, dtype=torch.float64)
        self._word_box = z(E, self.n_g_pad // 32, 4, dtype=torch.float32)    # acceleration data of the culled grid scan
        self._frame = z(E, 2, dtype=torch.float64)
        self.nearest_cell = z(E, n, dtype=torch.int32)
        # obs: the reference's [E, obs_dim, n_a], or [E, n_a, obs_dim] (agent-major rows, for device-side consumers)
        self.obs = z(E, self.obs_dim, n, dtype=out_dtype) if obs_layout == "reference" else z(E, n, self.obs_dim, dtype=out_dtype)
        self.reward = z(E, 1, n, dtype=out_dtype)
        self.done = z(E, 1, n, dtype=torch.bool)
        self._a_prior = [z(E, 2, n, dtype=out_dtype), z(E, 2, n, dtype=out_dtype)]
        self.neighbor_index = z(E, n, TOPO_NEI_MAX, dtype=torch.int32).fill_(-1)
        self.in_flags = z(E, n, dtype=torch.int32)
        if emit_indices:
            self.sensed_index = z(E, n, NUM_OBS_GRID_MAX, dtype=torch.int32).fill_(-1)
            self.occupied_index = z(E, n, NUM_OCC_GRID_MAX, dtype=torch.int32).fill_(-1)
        else:
            self.sensed_index = self.occupied_index = None

        buf = SwarmBuffers()
        buf.struct_size = C.sizeof(SwarmBuffers)
        buf.p, buf.dp, buf.grid = self.p.data_ptr(), self.dp.data_ptr(), self._grid.data_ptr()
        buf.n_g, buf.in_thresh = self._n_g.data_ptr(), self._in_thresh.data_ptr()
        buf.word_box, buf.frame = self._word_box.data_ptr(), self._frame.data_ptr()
        buf.nearest_cell = self.nearest_cell.data_ptr()
        buf.obs, buf.reward = self.obs.data_ptr(), self.reward.data_ptr()
        buf.a_prior[0], buf.a_prior[1] = self._a_prior[0].data_ptr(), self._a_prior[1].data_ptr()
        buf.neighbor_index, buf.in_flags = self.neighbor_index.data_ptr(), self.in_flags.data_ptr()
        if emit_indices:
            buf.sensed_index, buf.occupied_index = self.sensed_index.data_ptr(), self.occupied_index.data_ptr()
        self._buf = buf
        h = C.c_void_p()
        check(self.lib.swarm_create(C.byref(cfg), C.byref(buf), C.byref(h)), "swarm_create")
        self._h = h
        self.l_cell = np.zeros(E)
        self.n_g = np.zeros(E, dtype=np.int32)
        self.shapes_installed = False

    # ------------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.swarm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------------------------------------
    def set_grid(self, grid, n_g, l_cell, env0=0):
        """grid: [count, 2, n_g_max] float64 (numpy or CUDA tensor), each env's [2, n_g] grid_center stored
        contiguously at the start of its block (i.e. `block.reshape(-1)[:2*n_g].reshape(2, n_g)`);
        n_g, l_cell: [count] host arrays (assembly.py:163,179,187)."""
        n_g = np.ascontiguousarray(n_g, dtype=np.int32).reshape(-1)
        l_cell = np.ascontiguousarray(l_cell, dtype=np.float64).reshape(-1)
        count = n_g.shape[0]
        on_dev = isinstance(grid, torch.Tensor) and grid.is_cuda
        if on_dev:
            g = grid.to(torch.float64).contiguous()
            assert g.numel() == count * 2 * self.n_g_max
            ptr = g.data_ptr()
        else:
            g = np.ascontiguousarray(grid, dtype=np.float64)
            assert g.size == count * 2 * self.n_g_max, (g.shape, count, self.n_g_max)
            ptr = g.ctypes.data
        check(self.lib.swarm_set_grid(self._h, env0, count, C.c_void_p(ptr), int(on_dev), C.c_void_p(n_g.ctypes.data),
                                      C.c_void_p(l_cell.ctypes.data), self._stream()), "swarm_set_grid")
        self.n_g[env0:env0 + count] = n_g
        self.l_cell[env0:env0 + count] = l_cell

    def set_grid_pose(self, shape_ids, cos, sin, off_x, off_y, env0=0):
        """Target shapes as (library shape, pose): the device computes grid_center = R.origin + off itself (assembly.py:175-187,
        R = [[cos, sin], [-sin, cos]], products and sums rounded separately).  Needs set_shapes().  Same effect as set_grid with
        the grid `grid_from_pose` returns; the simulator then knows each pose exactly."""
        ids = np.ascontiguousarray(shape_ids, dtype=np.int32).reshape(-1)
        pose = np.ascontiguousarray(np.stack([np.broadcast_to(np.asarray(v, dtype=np.float64), ids.shape)
                                              for v in (cos, sin, off_x, off_y)], axis=1))
        check(self.lib.swarm_set_grid_pose(self._h, env0, ids.shape[0], C.c_void_p(ids.ctypes.data), C.c_void_p(pose.ctypes.data),
                                           self._stream()), "swarm_set_grid_pose")
        self.n_g[env0:env0 + ids.shape[0]] = self.shape_n_g[ids]
        self.l_cell[env0:env0 + ids.shape[0]] = self.shape_l_cells[ids]

    @staticmethod
    def grid_from_pose(origin, cos, sin, off_x, off_y):
        """The grid set_grid_pose installs for one env, computed on the host with the same roundings ([2, n_g] float64)."""
        return np.stack([(cos * origin[0] + sin * origin[1]) + off_x, ((-sin) * origin[0] + cos * origin[1]) + off_y])

    @staticmethod
    def pack_grids(grids, n_g_max):
        """list of [2, n_g] arrays -> ([count, 2*n_g_max] block array, n_g[count])"""
        out = np.zeros((len(grids), 2 * n_g_max))
        n_g = np.zeros(len(grids), dtype=np.int32)
        for k, g in enumerate(grids):
            g = np.ascontiguousarray(g, dtype=np.float64)
            out[k, :g.size] = g.reshape(-1)
            n_g[k] = g.shape[1]
        return out, n_g

    def set_shapes(self, grid_origins, l_cells):
        """Upload the shape library used by reset(): grid_origins is a list of [2, n_g] origin-frame grids (the transposed
        `grid_coords` of the reference's results.pkl, assembly.py:117,164), l_cells their cell sizes."""
        blocks, n_g = self.pack_grids(grid_origins, self.n_g_max)
        l_cells = np.ascontiguousarray(l_cells, dtype=np.float64)
        check(self.lib.swarm_set_shapes(self._h, len(grid_origins), C.c_void_p(blocks.ctypes.data), C.c_void_p(n_g.ctypes.data),
                                        C.c_void_p(l_cells.ctypes.data)), "swarm_set_shapes")
        self.shape_l_cells, self.shape_n_g = l_cells.copy(), n_g.copy()
        self.shapes_installed = True

    def reset(self, seed, episode=0, env_offset=0, env_mask=None):
        """reset() of assembly.py:156-223 for all envs (or those where env_mask is True) on the device, then the first
        observation.  Returns obs; `self.reset_info` [E, 8] holds {shape, cos, sin, off_x, off_y, wide-spawn flag, cluster_x, cluster_y}."""
        if not hasattr(self, "reset_info"):
            self.reset_info = torch.zeros(self.E, 8, dtype=torch.float64, device=self.device)
        mptr = None
        if env_mask is not None:
            env_mask = env_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            assert env_mask.numel() == self.E
            mptr = C.c_void_p(env_mask.data_ptr())
        check(self.lib.swarm_reset(self._h, int(seed), int(episode), int(env_offset), mptr,
                                   C.c_void_p(self.reset_info.data_ptr()), self._stream()), "swarm_reset")
        return self.obs

    def reset_envs(self, env_ids, seed, episode=0, env_offset=0):
        """reset() for the listed envs only (int32 CUDA tensor of distinct env ids): the auto-reset of a vector env."""
        assert env_ids.is_cuda and env_ids.dtype == torch.int32 and env_ids.is_contiguous()
        if not hasattr(self, "reset_info"):
            self.reset_info = torch.zeros(self.E, 8, dtype=torch.float64, device=self.device)
        check(self.lib.swarm_reset_envs(self._h, int(seed), int(episode), int(env_offset), C.c_void_p(env_ids.data_ptr()),
                                        int(env_ids.numel()), C.c_void_p(self.reset_info.data_ptr()), self._stream()), "swarm_reset_envs")
        return self.obs

    def measure_fma_peak(self):
        """(fp32, fp64) dense FMA TFLOP/s of this device, measured by a register-resident FMA loop."""
        a, b = C.c_double(), C.c_double()
        check(self.lib.swarm_measure_fma_peak(self.device.index, C.byref(a), C.byref(b)), "swarm_measure_fma_peak")
        return a.value, b.value

    def metrics(self):
        """[E, 3] float64 device tensor: coverage_rate, distribution_uniformity, voronoi_based_uniformity of every env
        (assembly_wrapper.py:48-129), computed on the device."""
        if not hasattr(self, "_metrics"):
            self._metrics = torch.zeros(self.E, 3, dtype=torch.float64, device=self.device)
        check(self.lib.swarm_metrics(self._h, C.c_void_p(self._metrics.data_ptr()), self._stream()), "swarm_metrics")
        return self._metrics

    def set_state(self, p, dp):
        """Overwrite positions / velocities ([E,2,n_a]); like assigning env.p / env.dp in the reference."""
        self.p.copy_(torch.as_tensor(p, dtype=torch.float64).reshape(self.E, 2, self.n_a))
        self.dp.copy_(torch.as_tensor(dp, dtype=torch.float64).reshape(self.E, 2, self.n_a))
        check(self.lib.swarm_mark_state_dirty(self._h), "swarm_mark_state_dirty")

    def strategy_actions(self, kind, out=None):
        """Actions of the reference env's own strategies for the current state: kind 'rule' (assembly.py:530-601) or 'llm'
        (assembly.py:524-529, 876-941).  [E, 2, n_a] float64 CUDA tensor; pass it to step() (float64 actions, assembly.py:633)."""
        k = {"rule": _lib.SWARM_STRATEGY_RULE, "llm": _lib.SWARM_STRATEGY_LLM}[kind]
        if out is None:
            out = torch.empty(self.E, 2, self.n_a, dtype=torch.float64, device=self.device)
        assert out.is_cuda and out.dtype == torch.float64 and out.is_contiguous() and out.numel() == self.E * 2 * self.n_a
        check(self.lib.swarm_strategy_actions(self._h, k, C.c_void_p(out.data_ptr()), self._stream()), "swarm_strategy_actions")
        return out

    def set_obs_buffer(self, obs):
        """Redirect the observation output of the following observe()/step() calls to `obs` (same shape / dtype, CUDA,
        contiguous); `self.obs` then refers to it.  Alternate two buffers to keep the previous observation without a copy."""
        assert obs.is_cuda and obs.is_contiguous() and obs.shape == self.obs.shape and obs.dtype == self.obs.dtype
        check(self.lib.swarm_set_obs_buffer(self._h, C.c_void_p(obs.data_ptr())), "swarm_set_obs_buffer")
        self.obs = obs

    def check_guards(self):
        """True iff every guard zone around the device buffers still holds its fill pattern (needs guard_bytes > 0)."""
        assert self._guards, "construct with guard_bytes > 0"
        ok = True
        for raw, gb, nbytes in self._guards:
            ok = ok and bool((raw[:gb] == 0xA5).all()) and bool((raw[gb + nbytes:] == 0xA5).all())
        return ok

    def mark_state_dirty(self):
        check(self.lib.swarm_mark_state_dirty(self._h), "swarm_mark_state_dirty")

    @property
    def fast_path(self):
        """0: the general culled scan runs next; 1: the lookup-scan kernel (shape library set, every env's grid recognised);
        2: lookup scan with exactly known poses (grids built by reset()): cells recomputed from the library."""
        return int(self.lib.swarm_fast_path(self._h))

    @property
    def observed(self):
        """True once an observation exists (observe / reset / restore_observation): step() needs its neighbour list."""
        return bool(self.lib.swarm_is_observed(self._h))

    def restore_observation(self):
        """State restore: the caller copied neighbor_index / in_flags / nearest_cell (and the outputs) of an earlier handle
        into this one's buffers; treat them as this handle's last observation (the next step computes its prior from them)."""
        check(self.lib.swarm_restore_observation(self._h), "swarm_restore_observation")

    # ------------------------------------------------------------------------------------------------
    def observe(self):
        """Tail of reset() (assembly.py:221): observation of the current state."""
        check(self.lib.swarm_observe(self._h, self._stream()), "swarm_observe")
        return self.obs

    def step(self, act):
        """act: CUDA tensor [E, 2, n_a], float32 or float64.  Returns the reference's 5-tuple (assembly.py:666)
        as device tensors; `info` is None."""
        if not (isinstance(act, torch.Tensor) and act.is_cuda):
            raise TypeError("step() takes a CUDA tensor; use step_host() for host buffers")
        if act.dtype not in (torch.float32, torch.float64):
            act = act.to(torch.float32)
        act = act.contiguous()
        assert act.numel() == self.E * 2 * self.n_a
        dt = _lib.SWARM_F32 if act.dtype == torch.float32 else _lib.SWARM_F64
        check(self.lib.swarm_step(self._h, C.c_void_p(act.data_ptr()), dt, self._stream()), "swarm_step")
        return self.obs, self.reward, self.done, None, (self.a_prior if self.want_prior else None)

    def step_host(self, act_host, obs_host=None, reward_host=None, a_prior_host=None):
        """Same step through host buffers (numpy / pinned torch CPU tensors): H2D actions, step, D2H results."""
        def ptr(a):
            if a is None:
                return None
            if isinstance(a, torch.Tensor):
                assert not a.is_cuda and a.is_contiguous()
                return C.c_void_p(a.data_ptr())
            assert a.flags["C_CONTIGUOUS"]
            return C.c_void_p(a.ctypes.data)
        if isinstance(act_host, np.ndarray):
            assert act_host.dtype == np.float32
        else:
            assert act_host.dtype == torch.float32
        check(self.lib.swarm_step_host(self._h, ptr(act_host), ptr(obs_host), ptr(reward_host), ptr(a_prior_host),
                                       self._stream()), "swarm_step_host")

    @property
    def a_prior(self):
        """a_prior returned by the most recent step (double-buffered on the device)."""
        ptr = self.lib.swarm_a_prior_ptr(self._h)
        return self._a_prior[0] if ptr == self._a_prior[0].data_ptr() else self._a_prior[1]

    def fill_actions(self, out, seed, step, env_offset=0):
        """Synthetic U(-1,1) float32 actions [E,2,n_a], identical to oracle.fill_actions for the same keys."""
        assert out.is_cuda and out.dtype == torch.float32 and out.numel() == self.E * 2 * self.n_a
        check(self.lib.swarm_fill_actions(self._h, seed, step, env_offset, C.c_void_p(out.data_ptr()), self._stream()),
              "swarm_fill_actions")
        return out

    @property
    def launch_count(self):
        return int(self.lib.swarm_launch_count(self._h))

    def kernel_geometry(self):
        t, s, c = C.c_int32(), C.c_int32(), C.c_int32()
        check(self.lib.swarm_kernel_geometry(self._h, C.byref(t), C.byref(s), C.byref(c)), "swarm_kernel_geometry")
        return dict(threads_per_cta=t.value, smem_bytes=s.value, ctas=c.value)

    # ------------------------------------------------------------------------------------------------
    def algorithmic_bytes_per_agent_step(self, mean_n_g=None, survey=True):
        """Unavoidable HBM traffic of one step per agent, for the roofline figure.  survey=True is SURVEY.md §8(d)'s count
        (read a, read + write p/dp, write obs, reward, done, a_prior, read the env's cells once: 1126 B for the production layout
        at n_g = 512, n_a = 30; + the four index arrays in the parity layout).  survey=False adds what this implementation also
        moves by design: neighbor_index / in_flags (the next prior reads them) and the nearest-cell seed."""
        osz = 4 if self.out_dtype == torch.float32 else 8
        ng = float(np.mean(self.n_g)) if mean_n_g is None else mean_n_g
        b = 2 * 4                      # read action (f32 x 2)
        b += 4 * 8 + 4 * 8             # read + write p, dp
        b += self.obs_dim * osz        # write obs
        b += osz + 1                   # write reward, done
        b += 2 * osz                   # write a_prior
        b += 2 * 8 * ng / self.n_a     # read the env's cell list once per env
        if self.emit_indices:
            b += (TOPO_NEI_MAX + 1 + NUM_OBS_GRID_MAX + NUM_OCC_GRID_MAX) * 4
        if not survey:
            b -= 1                     # done is constant False and never rewritten
            if not self.emit_indices:
                b += TOPO_NEI_MAX * 4 + 4
            b += 4 + 4                 # read + write nearest_cell (seed of the nearest-cell search)
            b += 2 * 8 * (math.ceil(ng / 32) * 32 - ng) / self.n_a
        return b
