"""ctypes binding of libmdpp_b200.so (the C ABI in include/mdpp_b200.h).

There is NO fallback: if the library is missing or a symbol is absent this
module raises, and every VectorRLToyEnv operation goes through it.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# MDPP_LIB: A/B timing of two builds (tools/); the default is the in-tree library
LIB_PATH = os.environ.get("MDPP_LIB") or os.path.join(HERE, "libmdpp_b200.so")

ABI_VERSION = 4  # MDPP_ABI_VERSION of include/mdpp_b200.h
MDPP_NOISE_OFF, MDPP_NOISE_REPLAY, MDPP_NOISE_PHILOX = 0, 1, 2
MDPP_N_STATS = 8
STATS_SLOTS = 64  # copies of the counter rows the kernels spread their atomics over
MDPP_NORMAL_F64, MDPP_NORMAL_FAST, MDPP_NORMAL_ZIGGURAT = 0, 1, 2
MDPP_OBS_I64, MDPP_OBS_I32, MDPP_OBS_U8 = 0, 1, 2
MDPP_REWARD_POINT, MDPP_REWARD_LINE = 0, 1
MDPP_LAUNCH_OVERLAP_PREVIOUS = 1
STAT_NAMES = ("episodes", "transitions", "reward", "noisy_transitions",
              "abs_reward_noise", "abs_transition_noise", "reserved",
              "terminated")

# every symbol include/mdpp_b200.h declares
EXPORTED_SYMBOLS = (
    "mdpp_abi_version", "mdpp_create", "mdpp_destroy", "mdpp_last_error",
    "mdpp_set_discrete_groups", "mdpp_discrete_rollout", "mdpp_discrete_reset",
    "mdpp_set_jit", "mdpp_jit_last_used", "mdpp_jit_log", "mdpp_jit_selftest",
    "mdpp_set_continuous_config", "mdpp_continuous_rollout",
    "mdpp_continuous_reset", "mdpp_render_discrete", "mdpp_render_continuous",
    "mdpp_set_grid_config", "mdpp_grid_rollout", "mdpp_grid_reset",
    "mdpp_ziggurat_tables",
    "mdpp_tail_actions", "mdpp_tail_post", "mdpp_tail_image_shift",
    "mdpp_set_continuous_groups",
    "mdpp_set_grid_groups",
    "mdpp_set_image_discrete_groups", "mdpp_render_discrete_groups",
    "mdpp_set_image_continuous_groups", "mdpp_render_continuous_groups",
    "mdpp_discrete_qlearn", "mdpp_grid_qlearn",
    "mdpp_continuous_ars", "mdpp_continuous_ars_update",
    "mdpp_continuous_ars_perturbations",
    "mdpp_discrete_qeval", "mdpp_grid_qeval", "mdpp_continuous_ars_eval",
)
MDPP_MAX_DIM, MDPP_MAX_ORDER, MDPP_MAX_TERM_BOXES = 16, 4, 8


def _ptr(t):
    """Device pointer of a tensor for a struct field or argument (NULL for None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


class DiscreteGroup(C.Structure):
    _fields_ = [
        ("n_states", C.c_int32), ("n_actions", C.c_int32),
        ("sequence_length", C.c_int32), ("delay", C.c_int32),
        ("reward_every_n_steps", C.c_int32), ("custom_reward", C.c_int32),
        ("n_sequences", C.c_int32), ("has_transition_noise", C.c_int32),
        ("has_reward_noise", C.c_int32), ("reserved0", C.c_int32),
        ("transition_noise", C.c_double), ("reward_noise_std", C.c_double),
        ("reward_scale", C.c_double), ("reward_shift", C.c_double),
        ("term_state_reward", C.c_double),
        ("transition", C.c_void_p), ("terminal", C.c_void_p),
        ("init_cdf", C.c_void_p), ("noise_cdf", C.c_void_p),
        ("sequences", C.c_void_p), ("sequence_rewards", C.c_void_p),
        ("reward_matrix", C.c_void_p),
        ("env_begin", C.c_int64), ("env_count", C.c_int64),
        ("global_id_base", C.c_int64),
        ("n_states_irr", C.c_int32), ("n_actions_irr", C.c_int32),
        ("transition_irr", C.c_void_p), ("init_cdf_irr", C.c_void_p),
        ("noise_cdf_irr", C.c_void_p),
    ]


class DiscreteState(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int64),
        ("cur_state", C.c_void_p), ("seq_key", C.c_void_p),
        ("t_episode", C.c_void_p), ("episode", C.c_void_p),
        ("ring", C.c_void_p),
        ("ring_depth", C.c_int32), ("history_depth", C.c_int32),
        ("history", C.c_void_p), ("stats", C.c_void_p),
        ("cur_state_irr", C.c_void_p),
        ("stats_slots", C.c_int32), ("reserved1", C.c_int32),
    ]


class DiscreteIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("obs", C.c_void_p), ("final_obs", C.c_void_p),
        ("reward", C.c_void_p), ("terminated", C.c_void_p),
        ("truncated", C.c_void_p), ("replay_transition_u", C.c_void_p),
        ("replay_reward_noise", C.c_void_p), ("replay_reset_u", C.c_void_p),
        ("obs_dtype", C.c_int32), ("reserved0", C.c_int32),
    ]


class StepOpts(C.Structure):
    _fields_ = [
        ("n_steps", C.c_int32), ("noise_mode", C.c_int32),
        ("autoreset", C.c_int32), ("horizon", C.c_int32),
        ("normal_mode", C.c_int32), ("flags", C.c_int32),
        ("seed", C.c_uint64), ("step_index", C.c_uint64),
        ("env_id_offset", C.c_int64), ("step_index_dev", C.c_void_p),
    ]


class QlearnParams(C.Structure):
    _fields_ = [
        ("alpha", C.c_double), ("gamma", C.c_double), ("epsilon", C.c_double),
        ("q", C.c_void_p), ("q_states", C.c_int32), ("q_actions", C.c_int32),
        ("ep_return", C.c_void_p), ("ret_sum", C.c_void_p),
        ("ret_count", C.c_void_p), ("actions_taken", C.c_void_p),
    ]


class ArsParams(C.Structure):
    _fields_ = [
        ("step_size", C.c_double), ("noise_std", C.c_double),
        ("theta", C.c_void_p), ("fitness", C.c_void_p),
        ("ep_return", C.c_void_p), ("ret_sum", C.c_void_p),
        ("ret_count", C.c_void_p), ("actions_taken", C.c_void_p),
        ("top_directions", C.c_int32), ("reserved0", C.c_int32),
        ("iteration", C.c_uint64), ("seed", C.c_uint64),
        ("env_id_offset", C.c_int64), ("delta_out", C.c_void_p),
        ("group_stats", C.c_void_p),
    ]


class EvalParams(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("q_states", C.c_int32), ("q_actions", C.c_int32),
        ("theta", C.c_void_p), ("episodes", C.c_int32), ("reserved0", C.c_int32),
        ("ret_sum", C.c_void_p), ("ret_count", C.c_void_p), ("len_sum", C.c_void_p),
    ]


class ContinuousConfig(C.Structure):
    _fields_ = [
        ("dim", C.c_int32), ("order", C.c_int32), ("n_relevant", C.c_int32),
        ("delay", C.c_int32), ("reward_every_n_steps", C.c_int32),
        ("dense", C.c_int32), ("has_transition_noise", C.c_int32),
        ("has_reward_noise", C.c_int32), ("image_mode", C.c_int32),
        ("target_is_f64", C.c_int32), ("n_term_boxes", C.c_int32),
        ("is_f64", C.c_int32),
        ("inertia", C.c_double), ("time_unit", C.c_double),
        ("state_space_max", C.c_double), ("action_space_max", C.c_double),
        ("target_radius", C.c_double), ("action_loss_weight", C.c_double),
        ("transition_noise_std", C.c_double), ("reward_noise_std", C.c_double),
        ("reward_scale", C.c_double), ("reward_shift", C.c_double),
        ("term_state_reward", C.c_double),
        ("relevant_indices", C.c_int32 * MDPP_MAX_DIM),
        ("target_point", C.c_double * MDPP_MAX_DIM),
        ("term_low", C.c_double * (MDPP_MAX_TERM_BOXES * MDPP_MAX_DIM)),
        ("term_high", C.c_double * (MDPP_MAX_TERM_BOXES * MDPP_MAX_DIM)),
        ("inertia_mode", C.c_int32), ("reward_kind", C.c_int32),
        ("inertia_vec", C.c_double * MDPP_MAX_DIM),
        ("sequence_length", C.c_int32), ("reserved_cfg", C.c_int32),
    ]


class ContinuousGroup(C.Structure):
    _fields_ = [("cfg", ContinuousConfig), ("env_begin", C.c_int64),
                ("env_count", C.c_int64), ("global_id_base", C.c_int64)]


class ContinuousState(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int64), ("derivs", C.c_void_p), ("emitted", C.c_void_p),
        ("t_episode", C.c_void_p), ("episode", C.c_void_p),
        ("reached", C.c_void_p), ("ring", C.c_void_p), ("stats", C.c_void_p),
        ("stats_slots", C.c_int32), ("reserved1", C.c_int32),
        ("hist", C.c_void_p),
    ]


class ContinuousIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("obs", C.c_void_p), ("final_obs", C.c_void_p),
        ("reward", C.c_void_p), ("terminated", C.c_void_p),
        ("truncated", C.c_void_p), ("replay_state_noise", C.c_void_p),
        ("replay_reward_noise", C.c_void_p), ("replay_reset_state", C.c_void_p),
    ]


class ImageDiscreteTables(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("n_states", C.c_int32),
        ("r_min", C.c_int32), ("n_radii", C.c_int32),
        ("n_xvar", C.c_int32), ("n_yvar", C.c_int32),
        ("has_scale", C.c_int32), ("has_shift", C.c_int32),
        ("has_rotate", C.c_int32), ("has_flip", C.c_int32),
        ("sh_quant", C.c_int32), ("ro_quant", C.c_int32),
        ("n_sub_images", C.c_int32),
        ("mask_bits", C.c_void_p), ("mask_index", C.c_void_p),
        ("xvar", C.c_void_p), ("yvar", C.c_void_p), ("rot_coeff", C.c_void_p),
        ("r_thresholds", C.c_void_p),
    ]


class ImageDiscreteGroup(C.Structure):
    _fields_ = [("tb", ImageDiscreteTables), ("env_begin", C.c_int64),
                ("env_count", C.c_int64), ("global_id_base", C.c_int64)]


MDPP_MAX_STAMP_ROWS = 32


class ImageContinuousConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("dim", C.c_int32),
        ("n_sub_images", C.c_int32),
        ("rel_index", C.c_int32 * 2), ("irr_index", C.c_int32 * 2),
        ("is_f64", C.c_int32), ("n_rects", C.c_int32), ("has_target", C.c_int32),
        ("stamp_rows", C.c_int32), ("stamp_radius", C.c_int32),
        ("reserved0", C.c_int32),
        ("feat_low", C.c_double * 2), ("feat_high", C.c_double * 2),
        ("rect", (C.c_int32 * 4) * MDPP_MAX_TERM_BOXES),
        ("target_pixel", C.c_int32 * 2),
        ("stamp", (C.c_int32 * 2) * MDPP_MAX_STAMP_ROWS),
        ("vline", (C.c_uint64 * 4) * 2), ("hline", (C.c_uint64 * 4) * 2),
    ]


class ImageContinuousGroup(C.Structure):
    _fields_ = [("cfg", ImageContinuousConfig), ("env_begin", C.c_int64),
                ("env_count", C.c_int64)]


MDPP_MAX_GRID_DIMS = 4


class GridConfig(C.Structure):
    _fields_ = [
        ("n_dims", C.c_int32), ("dense", C.c_int32),
        ("reward_every_n_steps", C.c_int32),
        ("has_transition_noise", C.c_int32), ("has_reward_noise", C.c_int32),
        ("reserved0", C.c_int32),
        ("shape", C.c_int32 * MDPP_MAX_GRID_DIMS), ("target", C.c_int32 * 2),
        ("transition_noise", C.c_double), ("reward_noise_std", C.c_double),
        ("reward_scale", C.c_double), ("reward_shift", C.c_double),
        ("term_state_reward", C.c_double),
    ]


class GridGroup(C.Structure):
    _fields_ = [("cfg", GridConfig), ("env_begin", C.c_int64),
                ("env_count", C.c_int64), ("global_id_base", C.c_int64)]


class GridState(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int64), ("pos", C.c_void_p), ("t_episode", C.c_void_p),
        ("episode", C.c_void_p), ("reached", C.c_void_p), ("stats", C.c_void_p),
        ("stats_slots", C.c_int32), ("reserved1", C.c_int32),
        ("prev", C.c_void_p),
    ]


class GridIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("obs", C.c_void_p), ("final_obs", C.c_void_p),
        ("reward", C.c_void_p), ("terminated", C.c_void_p),
        ("truncated", C.c_void_p), ("replay_noise_u", C.c_void_p),
        ("replay_noise_action", C.c_void_p),
        ("replay_reward_noise", C.c_void_p), ("replay_reset_state", C.c_void_p),
    ]


class TailConfig(C.Structure):
    _fields_ = [
        ("discrete", C.c_int32), ("n_actions", C.c_int32), ("obs_dim", C.c_int32),
        ("obs_is_f64", C.c_int32), ("delay", C.c_int32),
        ("has_transition_noise", C.c_int32), ("has_reward_noise", C.c_int32),
        ("image_side", C.c_int32), ("image_channels", C.c_int32),
        ("image_padding", C.c_int32), ("sh_quant", C.c_int32),
        ("has_shift", C.c_int32),
        ("transition_noise", C.c_double), ("reward_noise_std", C.c_double),
        ("reward_scale", C.c_double), ("reward_shift", C.c_double),
        ("term_state_reward", C.c_double),
    ]


class TailState(C.Structure):
    _fields_ = [("n_envs", C.c_int64), ("ring", C.c_void_p),
                ("t_episode", C.c_void_p)]


_lib = None


def load():
    """Load the library once; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. "
            "Run `python -m mdp_playground_b200.build` (needs nvcc). There is "
            "no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTED_SYMBOLS:
        if not hasattr(lib, name):
            raise RuntimeError(f"{LIB_PATH} does not export {name}")
    P = C.c_void_p
    lib.mdpp_abi_version.restype = C.c_int
    lib.mdpp_create.argtypes = [C.c_int, C.POINTER(P)]
    lib.mdpp_destroy.argtypes = [P]
    lib.mdpp_destroy.restype = None
    lib.mdpp_last_error.argtypes = [P]
    lib.mdpp_last_error.restype = C.c_char_p
    lib.mdpp_set_discrete_groups.argtypes = [P, C.POINTER(DiscreteGroup), C.c_int32]
    lib.mdpp_discrete_rollout.argtypes = [
        P, C.POINTER(DiscreteState), C.POINTER(DiscreteIO), C.POINTER(StepOpts), P]
    lib.mdpp_discrete_qlearn.argtypes = [
        P, C.POINTER(DiscreteState), C.POINTER(DiscreteIO), C.POINTER(QlearnParams),
        C.POINTER(StepOpts), P]
    lib.mdpp_discrete_reset.argtypes = [
        P, C.POINTER(DiscreteState), P, P, P, P, C.POINTER(StepOpts), P]
    lib.mdpp_set_jit.argtypes = [P, C.c_int]
    lib.mdpp_ziggurat_tables.argtypes = [C.POINTER(P), C.POINTER(P), C.POINTER(P)]
    lib.mdpp_ziggurat_tables.restype = None
    lib.mdpp_set_jit.restype = None
    lib.mdpp_jit_last_used.argtypes = [P]
    lib.mdpp_jit_log.argtypes = [P]
    lib.mdpp_jit_log.restype = C.c_char_p
    lib.mdpp_jit_selftest.argtypes = [C.c_char_p, C.c_int]
    lib.mdpp_set_continuous_config.argtypes = [P, C.POINTER(ContinuousConfig)]
    lib.mdpp_set_continuous_groups.argtypes = [P, C.POINTER(ContinuousGroup), C.c_int32]
    lib.mdpp_continuous_rollout.argtypes = [
        P, C.POINTER(ContinuousState), C.POINTER(ContinuousIO),
        C.POINTER(StepOpts), P]
    lib.mdpp_continuous_ars.argtypes = [
        P, C.POINTER(ContinuousState), C.POINTER(ContinuousIO), C.POINTER(ArsParams),
        C.POINTER(StepOpts), P]
    lib.mdpp_continuous_ars_eval.argtypes = [
        P, C.POINTER(ContinuousState), C.POINTER(ContinuousIO), C.POINTER(EvalParams),
        C.POINTER(StepOpts), P]
    lib.mdpp_discrete_qeval.argtypes = [
        P, C.POINTER(DiscreteState), C.POINTER(DiscreteIO), C.POINTER(EvalParams),
        C.POINTER(StepOpts), P]
    lib.mdpp_grid_qeval.argtypes = [
        P, C.POINTER(GridState), C.POINTER(GridIO), C.POINTER(EvalParams),
        C.POINTER(StepOpts), P]
    lib.mdpp_continuous_ars_update.argtypes = [P, C.c_int64, C.POINTER(ArsParams), P]
    lib.mdpp_continuous_ars_perturbations.argtypes = [
        P, C.c_int64, C.POINTER(ArsParams), P]
    lib.mdpp_continuous_reset.argtypes = [
        P, C.POINTER(ContinuousState), P, P, P, C.POINTER(StepOpts), P]
    lib.mdpp_render_discrete.argtypes = [
        P, C.POINTER(ImageDiscreteTables), P, P, P, P, C.c_int64, C.c_int64,
        C.c_int32, C.POINTER(StepOpts), P]
    lib.mdpp_render_continuous.argtypes = [
        P, C.POINTER(ImageContinuousConfig), P, P, C.c_int64, P]
    lib.mdpp_set_image_discrete_groups.argtypes = [
        P, C.POINTER(ImageDiscreteGroup), C.c_int32]
    lib.mdpp_render_discrete_groups.argtypes = [
        P, P, P, P, P, C.c_int64, C.c_int64, C.c_int32, C.POINTER(StepOpts), P]
    lib.mdpp_set_image_continuous_groups.argtypes = [
        P, C.POINTER(ImageContinuousGroup), C.c_int32]
    lib.mdpp_render_continuous_groups.argtypes = [P, P, P, C.c_int64, C.c_int64, P]
    lib.mdpp_set_grid_config.argtypes = [P, C.POINTER(GridConfig)]
    lib.mdpp_set_grid_groups.argtypes = [P, C.POINTER(GridGroup), C.c_int32]
    lib.mdpp_grid_rollout.argtypes = [
        P, C.POINTER(GridState), C.POINTER(GridIO), C.POINTER(StepOpts), P]
    lib.mdpp_grid_qlearn.argtypes = [
        P, C.POINTER(GridState), C.POINTER(GridIO), C.POINTER(QlearnParams),
        C.POINTER(StepOpts), P]
    lib.mdpp_grid_reset.argtypes = [
        P, C.POINTER(GridState), P, P, P, C.POINTER(StepOpts), P]
    lib.mdpp_tail_actions.argtypes = [
        P, C.POINTER(TailConfig), P, P, P, C.c_int64, C.POINTER(StepOpts), P]
    lib.mdpp_tail_post.argtypes = [
        P, C.POINTER(TailConfig), C.POINTER(TailState), P, P, P, P, P, P, P,
        C.POINTER(StepOpts), P]
    lib.mdpp_tail_image_shift.argtypes = [
        P, C.POINTER(TailConfig), P, P, P, P, C.c_int64, C.POINTER(StepOpts), P]
    if lib.mdpp_abi_version() != ABI_VERSION:
        raise RuntimeError("libmdpp_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


class MdppError(RuntimeError):
    pass


def check(lib, ctx, rc):
    if rc != 0:
        msg = lib.mdpp_last_error(ctx)
        raise MdppError(f"libmdpp_b200 error {rc}: "
                        f"{msg.decode() if msg else '?'}")
