"""ctypes binding of include/swarm_b200.h.  Fails loudly when the CUDA library is missing: there is no
CPU implementation to fall back to."""
import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SWARM_B200_LIB") or os.path.join(PKG, "lib", "libswarm_b200.so")   # override: A/B builds

SWARM_OK, SWARM_ERR_INVALID, SWARM_ERR_UNSUPPORTED, SWARM_ERR_CUDA, SWARM_ERR_NO_DEVICE = range(5)
SWARM_F64, SWARM_F32 = 0, 1
SWARM_OBS_REFERENCE, SWARM_OBS_AGENT_MAJOR = 0, 1
SWARM_VARIANT_ASSEMBLY, SWARM_VARIANT_FLOCKING = 0, 1
SWARM_STRATEGY_RULE, SWARM_STRATEGY_LLM = 1, 2


class SwarmConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("device", C.c_int32), ("num_envs", C.c_int32), ("n_a", C.c_int32),
        ("n_g_max", C.c_int32), ("topo_nei_max", C.c_int32), ("num_obs_grid_max", C.c_int32),
        ("num_occupied_grid_max", C.c_int32), ("is_con_self_state", C.c_int32), ("is_periodic", C.c_int32),
        ("want_prior", C.c_int32), ("out_dtype", C.c_int32), ("emit_indices", C.c_int32),
        ("exact_occupancy", C.c_int32), ("brute_force_scan", C.c_int32), ("debug_flags", C.c_int32), ("obs_layout", C.c_int32), ("variant", C.c_int32),
        ("d_sen", C.c_double), ("r_avoid", C.c_double), ("size_a", C.c_double),
        ("k_ball", C.c_double), ("k_wall", C.c_double), ("c_wall", C.c_double),
        ("dt", C.c_double), ("vel_max", C.c_double), ("mass", C.c_double),
        ("boundary_pos", C.c_double * 4),
    ]


class SwarmBuffers(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("pad_", C.c_int32),
        ("p", C.c_void_p), ("dp", C.c_void_p), ("grid", C.c_void_p), ("n_g", C.c_void_p),
        ("word_box", C.c_void_p), ("frame", C.c_void_p),
        ("in_thresh", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p),
        ("a_prior", C.c_void_p * 2),
        ("neighbor_index", C.c_void_p), ("in_flags", C.c_void_p), ("nearest_cell", C.c_void_p),
        ("sensed_index", C.c_void_p), ("occupied_index", C.c_void_p),
    ]


SWARM_RENDER_CELLS, SWARM_RENDER_AGENTS, SWARM_RENDER_TRAILS = 1, 2, 4


class SwarmRenderArgs(C.Structure):        # swarm_render_args
    _fields_ = [
        ("struct_size", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("flags", C.c_int32), ("count", C.c_int32),
        ("pad_", C.c_int32), ("env_ids", C.c_void_p), ("view", C.c_double * 4), ("trail", C.c_void_p), ("trail_cap", C.c_int32),
        ("trail_len", C.c_int32), ("trail_head", C.c_int32), ("pad2_", C.c_int32), ("frames", C.c_void_p),
    ]


SWARM_PP_INPUT, SWARM_PP_STATIC, SWARM_PP_RANDOM, SWARM_PP_NEAREST = 0, 1, 2, 3


class SwarmPPConfig(C.Structure):          # swarm_pp_config (include/swarm_b200.h)
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("num_envs", C.c_int32), ("n_p", C.c_int32), ("n_e", C.c_int32),
        ("is_con_self_state", C.c_int32), ("is_periodic", C.c_int32), ("billiards", C.c_int32), ("out_dtype", C.c_int32),
        ("strategy_p", C.c_int32), ("strategy_e", C.c_int32),
        ("d_sen", C.c_double), ("size_a", C.c_double), ("k_ball", C.c_double), ("k_wall", C.c_double), ("c_wall", C.c_double),
        ("dt", C.c_double), ("vel_max_p", C.c_double), ("vel_max_e", C.c_double), ("mass", C.c_double),
        ("boundary_pos", C.c_double * 4), ("seed", C.c_uint64),
    ]


class SwarmPPBuffers(C.Structure):         # swarm_pp_buffers
    _fields_ = [("struct_size", C.c_uint32), ("p", C.c_void_p), ("dp", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p),
                ("neighbor_index", C.c_void_p)]


# every symbol include/swarm_b200.h declares (tests check the library exports all of them)
LEGACY_SYMBOLS = ["_get_observation", "_get_reward", "_sf_b2b_all", "_get_dist_b2w", "calculateActionPrior"]
BATCHED_SYMBOLS = ["swarm_grid_pad", "swarm_obs_dim", "swarm_create", "swarm_destroy", "swarm_set_grid",
                   "swarm_set_shapes", "swarm_reset", "swarm_metrics", "swarm_set_obs_buffer", "swarm_strategy_actions",
                   "swarm_mark_state_dirty", "swarm_observe", "swarm_step", "swarm_step_host", "swarm_a_prior_ptr",
                   "swarm_fill_actions", "swarm_launch_count", "swarm_kernel_geometry", "swarm_last_error",
                   "swarm_abi_version", "swarm_sqrt_threshold", "swarm_debug_rho", "swarm_restore_observation", "swarm_is_observed", "swarm_reset_envs", "swarm_measure_fma_peak", "swarm_fast_path", "swarm_set_grid_pose", "swarm_flock_observe", "swarm_flock_step", "swarm_selftest_division", "swarm_pp_obs_dim", "swarm_pp_observe", "swarm_pp_step",
                   "swarm_render", "swarm_render_palette",
                   "swarm_state_store_create", "swarm_state_store_destroy", "swarm_state_slot_bytes", "swarm_state_save", "swarm_state_load",
                   "swarm_prior_compile", "swarm_prior_program_create", "swarm_prior_program_destroy", "swarm_set_prior_program",
                   "swarm_prior_program_actions", "swarm_prior_population_create", "swarm_prior_population_destroy",
                   "swarm_set_prior_population", "swarm_prior_population_actions"]
ROLLOUT_SYMBOLS = ["swarm_rollout_push", "swarm_rollout_gather", "swarm_rollout_push_parts", "swarm_rollout_gather_ring"]
SWARM_PUSH_OBS, SWARM_PUSH_NEXT_OBS, SWARM_PUSH_SMALL = 1, 2, 4
POLICY_SYMBOLS = ["swarm_policy_create", "swarm_policy_destroy", "swarm_policy_load", "swarm_policy_step", "swarm_policy_launch_count",
                  "swarm_policy_set_precision", "swarm_policy_debug_buffer", "swarm_policy_rows_out", "swarm_policy_obs_layout"]
SWARM_POLICY_FP32, SWARM_POLICY_F16_TC, SWARM_POLICY_F16X3_TC = 0, 1, 2


class SwarmRolloutBuffers(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("pad_", C.c_int32),
        ("capacity", C.c_int64),
        ("obs", C.c_void_p), ("act", C.c_void_p), ("act_prior", C.c_void_p), ("log_pi", C.c_void_p),
        ("rew", C.c_void_p), ("next_obs", C.c_void_p), ("done", C.c_void_p),
    ]

_lib = None


class SwarmError(RuntimeError):
    pass


def load():
    """Loads the CUDA library (building is a separate, explicit step: marl_llm_b200.build.build_library)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise SwarmError(f"{LIB_PATH} is missing: build it with `python -m marl_llm_b200.build` "
                         "(needs nvcc; the simulator has no CPU fallback)")
    lib = C.CDLL(LIB_PATH, C.RTLD_GLOBAL)
    lib.swarm_last_error.restype = C.c_char_p
    lib.swarm_a_prior_ptr.restype = C.c_void_p
    lib.swarm_a_prior_ptr.argtypes = [C.c_void_p]
    lib.swarm_launch_count.restype = C.c_int64
    lib.swarm_launch_count.argtypes = [C.c_void_p]
    lib.swarm_create.argtypes = [C.POINTER(SwarmConfig), C.POINTER(SwarmBuffers), C.POINTER(C.c_void_p)]
    lib.swarm_destroy.argtypes = [C.c_void_p]
    lib.swarm_set_grid.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_mark_state_dirty.argtypes = [C.c_void_p]
    lib.swarm_fast_path.argtypes = [C.c_void_p]
    lib.swarm_flock_observe.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_flock_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.swarm_set_grid_pose.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_restore_observation.argtypes = [C.c_void_p]
    lib.swarm_is_observed.argtypes = [C.c_void_p]
    lib.swarm_set_obs_buffer.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_strategy_actions.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.swarm_metrics.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_render.argtypes = [C.c_void_p, C.POINTER(SwarmRenderArgs), C.c_void_p]
    lib.swarm_render_palette.argtypes = [C.c_void_p]
    lib.swarm_state_store_create.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
    lib.swarm_state_store_destroy.argtypes = [C.c_void_p]
    lib.swarm_state_slot_bytes.restype = C.c_int64
    lib.swarm_state_slot_bytes.argtypes = [C.c_void_p]
    lib.swarm_state_save.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.swarm_state_load.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.swarm_prior_compile.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.c_char_p, C.c_int64]
    lib.swarm_prior_program_create.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
    lib.swarm_prior_program_destroy.argtypes = [C.c_void_p]
    lib.swarm_set_prior_program.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_prior_program_actions.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_prior_population_create.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.swarm_prior_population_destroy.argtypes = [C.c_void_p]
    lib.swarm_set_prior_population.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_prior_population_actions.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_set_shapes.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_reset.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_reset_envs.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.swarm_measure_fma_peak.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.swarm_observe.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.swarm_step_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.swarm_fill_actions.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.swarm_kernel_geometry.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.swarm_grid_pad.argtypes = [C.c_int32]
    lib.swarm_obs_dim.argtypes = [C.POINTER(SwarmConfig)]
    lib.swarm_rollout_push.argtypes = [C.POINTER(SwarmRolloutBuffers), C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                       C.c_void_p, C.c_void_p]
    lib.swarm_rollout_gather.argtypes = [C.POINTER(SwarmRolloutBuffers), C.c_void_p, C.c_int32] + [C.c_void_p] * 8
    lib.swarm_rollout_push_parts.argtypes = [C.POINTER(SwarmRolloutBuffers), C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                             C.c_void_p, C.c_int, C.c_void_p]
    lib.swarm_rollout_gather_ring.argtypes = [C.POINTER(SwarmRolloutBuffers), C.c_void_p, C.c_int32, C.c_int64] + [C.c_void_p] * 8
    lib.swarm_policy_rows_out.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_policy_obs_layout.argtypes = [C.c_void_p, C.c_int]
    lib.swarm_policy_create.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    lib.swarm_policy_destroy.argtypes = [C.c_void_p]
    lib.swarm_policy_load.argtypes = [C.c_void_p] + [C.c_void_p] * 8
    lib.swarm_policy_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                      C.c_uint64, C.c_uint64, C.c_void_p]
    lib.swarm_policy_set_precision.argtypes = [C.c_void_p, C.c_int]
    lib.swarm_policy_debug_buffer.argtypes = [C.c_void_p, C.c_void_p]
    lib.swarm_policy_launch_count.restype = C.c_int64
    lib.swarm_policy_launch_count.argtypes = [C.c_void_p]
    lib.swarm_debug_rho.argtypes = [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]
    lib.swarm_pp_obs_dim.argtypes = [C.POINTER(SwarmPPConfig)]
    lib.swarm_pp_observe.argtypes = [C.POINTER(SwarmPPConfig), C.POINTER(SwarmPPBuffers), C.c_void_p]
    lib.swarm_pp_step.argtypes = [C.POINTER(SwarmPPConfig), C.POINTER(SwarmPPBuffers), C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p]
    lib.swarm_selftest_division.argtypes = [C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, C.POINTER(C.c_uint64)]
    lib.swarm_sqrt_threshold.restype = C.c_double
    lib.swarm_sqrt_threshold.argtypes = [C.c_double, C.c_int]
    _lib = lib
    return lib


def check(rc, what):
    if rc != SWARM_OK:
        msg = load().swarm_last_error().decode("utf-8", "replace")
        raise SwarmError(f"{what} failed (code {rc}): {msg}")
