"""Config-dict handling for VectorRLToyEnv: same keys, defaults and checks as
the reference constructor (rl_toy_env.py:216-666; key list in SURVEY.md
appendix B).  Unknown keys are accepted and ignored, as in the reference."""
import sys
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional

import numpy as np


def np_random(seed):
    """gymnasium.utils.seeding.np_random as used at rl_toy_env.py:2399."""
    if seed is not None and not (isinstance(seed, int) and seed >= 0):
        raise ValueError(f"seed must be a non-negative python int, got {seed!r}")
    ss = np.random.SeedSequence(seed)
    return np.random.Generator(np.random.PCG64(ss)), ss.entropy


_SEED_KEYS = ("relevant_state_space", "relevant_action_space",
              "irrelevant_state_space", "irrelevant_action_space",
              "state_space", "action_space", "image_representations")


@dataclass
class EnvSpec:
    """Everything the kernels and table builders need, with defaults filled."""
    config: Dict[str, Any]
    kind: str = "discrete"
    seed_dict: Dict[str, Any] = field(default_factory=dict)
    env_rng: Any = None  # E stream after the seed fan-out (used by table gen)
    use_custom_mdp: bool = False
    terminal_state_density: float = 0.25
    term_state_reward: float = 0.0
    delay: int = 0
    sequence_length: int = 1
    reward_density: float = 0.25
    make_denser: bool = False
    maximally_connected: bool = True
    has_reward_noise: bool = False
    reward_noise_std: float = 0.0
    has_transition_noise: bool = False
    transition_noise: float = 0.0
    reward_scale: float = 1.0
    reward_shift: float = 0.0
    image_representations: bool = False
    image_transforms: str = "none"
    image_width: int = 100
    image_height: int = 100
    image_sh_quant: Optional[int] = None
    image_ro_quant: Optional[int] = None
    image_scale_range: Optional[tuple] = None
    reward_every_n_steps: int = 1
    repeats_in_sequences: bool = False
    action_loss_weight: float = 0.0
    # discrete
    reward_dist: Any = None
    diameter: int = 1
    action_space_size: int = 0
    state_space_size: int = 0
    irrelevant_features: bool = False  # discrete: a second, reward-free sub-MDP
    action_space_size_irr: int = 0
    state_space_size_irr: int = 0
    dtype_s: Any = None
    dtype_o: Any = None
    # continuous
    state_space_dim: int = 0
    dynamics_order: int = 1
    inertia: float = 1.0
    time_unit: float = 1.0
    target_radius: float = 0.05
    relevant_indices: List[int] = field(default_factory=list)
    target_point: Any = None
    reward_function: str = "move_to_a_point"
    state_space_max: float = float("inf")
    action_space_max: float = float("inf")
    terminal_centres: Any = None
    term_state_edge: float = 0.0
    # grid
    grid_shape: tuple = ()
    terminal_cells: Any = None


def state_space_kind(config):
    """"discrete", "continuous" or "grid": the config's state_space_type,
    lower-cased; {} is the reference's default discrete config (:227-235)."""
    if config == {}:
        return "discrete"
    kind = config["state_space_type"].lower()
    if kind not in ("discrete", "continuous", "grid"):
        raise ValueError("Unknown state_space_type")
    return kind


def parse_config(config):
    """Fill defaults exactly like RLToyEnv.__init__ (:227-666)."""
    if config == {}:  # :227-235
        config = dict(state_space_size=8, action_space_size=8,
                      state_space_type="discrete", action_space_type="discrete",
                      terminal_state_density=0.25, maximally_connected=True)
    sp = EnvSpec(config=config)
    # ---- seed fan-out :285-334 -------------------------------------------
    if "seed" in config and isinstance(config["seed"], dict):
        sp.seed_dict = config["seed"]
        sp.env_rng, _ = np_random(sp.seed_dict["env"])
    else:
        seed_int = config.get("seed")
        if seed_int is not None and not isinstance(seed_int, int):
            raise TypeError("Unsupported data type for seed", type(seed_int))
        sp.env_rng, _ = np_random(seed_int)
        sp.seed_dict = {"env": seed_int}
        for k in _SEED_KEYS:
            sp.seed_dict[k] = sp.env_rng.integers(sys.maxsize).item()

    kind = sp.kind = config["state_space_type"] = state_space_kind(config)
    g = config.get
    sp.use_custom_mdp = bool(g("use_custom_mdp", False))
    if sp.use_custom_mdp:
        assert "transition_function" in config
        assert "reward_function" in config
    sp.terminal_state_density = g("terminal_state_density", 0.25)
    sp.term_state_reward = float(g("term_state_reward", 0.0))
    sp.delay = int(g("delay", 0))
    sp.sequence_length = int(g("sequence_length", 1))
    sp.reward_density = g("reward_density", 0.25)
    sp.make_denser = bool(g("make_denser", kind == "continuous"))
    sp.maximally_connected = bool(g("maximally_connected", True))
    for key in ("reward_noise", "transition_noise"):
        if callable(g(key)):
            raise NotImplementedError(
                f"callable {key} cannot run on the device; pass a float "
                "(or use noise='replay' with your own draws)")
    sp.has_reward_noise = "reward_noise" in config and g("reward_noise") is not None
    sp.reward_noise_std = float(g("reward_noise") or 0.0)
    sp.has_transition_noise = ("transition_noise" in config
                               and g("transition_noise") is not None)
    sp.transition_noise = float(g("transition_noise") or 0.0)
    sp.reward_scale = float(g("reward_scale", 1.0))
    sp.reward_shift = float(g("reward_shift", 0.0))
    sp.irrelevant_features = bool(g("irrelevant_features", False))
    sp.image_representations = bool(g("image_representations", False))
    if "image_transforms" in config:
        assert kind == "discrete", \
            "Image transforms are only applicable to discrete envs."
        sp.image_transforms = config["image_transforms"]
    sp.image_width = int(g("image_width", 100))
    sp.image_height = int(g("image_height", 100))
    if kind == "discrete":
        tr = sp.image_transforms
        sp.image_sh_quant = g("image_sh_quant", 1 if "shift" in tr else None)
        sp.image_ro_quant = g("image_ro_quant", 1 if "rotate" in tr else None)
        sp.image_scale_range = g("image_scale_range",
                                 (0.5, 1.5) if "scale" in tr else None)
        sp.reward_dist = g("reward_dist", None)
        if callable(sp.reward_dist):
            raise NotImplementedError("callable reward_dist is not supported")
        sp.diameter = int(g("diameter", 1))
    elif kind == "grid":  # :539-541, :655-657
        assert "grid_shape" in config
        sp.grid_shape = tuple(int(n) for n in config["grid_shape"])
        assert len(sp.grid_shape) == 2, "grid_shape must be 2-D"
        if config["reward_function"] != "move_to_a_point":
            raise NotImplementedError("grid: only move_to_a_point (as in the reference)")
        sp.target_point = [int(v) for v in config["target_point"]]
        if "make_denser" not in config:
            # the reference leaves the attribute unset for grid envs (:384-390)
            # and raises AttributeError in the first reward computation
            raise ValueError("grid environments need an explicit make_denser")
        if sp.delay != 0 or sp.sequence_length != 1:
            # np.array(augmented_state) is ragged then (:1950): the reference
            # raises ValueError in the first step
            raise NotImplementedError(
                "grid environments: delay must be 0 and sequence_length 1 "
                "(anything else crashes in the reference)")
        if sp.irrelevant_features:
            sp.grid_shape = sp.grid_shape * 2  # :604-608
        if callable(config.get("terminal_states")):
            raise NotImplementedError("callable terminal_states")
        # terminal cells never end an episode in the reference (SURVEY 8f N1
        # probe); they are drawn in image observations
        sp.terminal_cells = [[int(v) for v in c]
                             for c in config.get("terminal_states", [])]
    else:
        sp.state_space_dim = int(config["state_space_dim"])
        config.setdefault("reward_function", "move_to_a_point")
        if config["reward_function"] not in ("move_to_a_point", "move_along_a_line"):
            raise ValueError("unknown reward_function " + str(config["reward_function"]))
        sp.reward_function = config["reward_function"]
        sp.dynamics_order = int(g("transition_dynamics_order", 1))
        sp.inertia = g("inertia", 1.0)
        sp.time_unit = g("time_unit", 1.0)
        sp.target_radius = g("target_radius", 0.05)
    sp.action_loss_weight = g("action_loss_weight", 0.0)
    if "reward_every_n_steps" in config:
        sp.reward_every_n_steps = int(config["reward_every_n_steps"])
    else:  # :550-561
        sp.reward_every_n_steps = sp.sequence_length if kind == "discrete" else 1
    sp.repeats_in_sequences = bool(g("repeats_in_sequences", False))

    if kind == "discrete":  # :570-591
        sp.dtype_s = g("dtype_s", np.int64)
        if sp.irrelevant_features:  # :574-578, sizes are [relevant, irrelevant]
            assert len(config["action_space_size"]) == 2, (
                "Currently, 1st sub-state (and action) space is assumed to be "
                "relevant to rewards and 2nd one is irrelevant. Please provide "
                "a list with sizes for the 2.")
            if sp.use_custom_mdp:
                raise NotImplementedError(
                    "irrelevant_features with use_custom_mdp")
            sp.action_space_size = int(config["action_space_size"][0])
            sp.action_space_size_irr = int(config["action_space_size"][1])
            sp.state_space_size_irr = sp.action_space_size_irr * sp.diameter
        else:
            assert isinstance(config["action_space_size"], int), (
                "Did you mean to turn irrelevant_features? If not, please "
                "provide an int for action_space_size.")
            sp.action_space_size = config["action_space_size"]
        if sp.use_custom_mdp:
            sp.state_space_size = int(config["state_space_size"])
        else:
            sp.state_space_size = sp.action_space_size * sp.diameter
    elif kind == "grid":
        sp.dtype_s = g("dtype_s", np.int64)
        if np.dtype(sp.dtype_s) != np.dtype(np.int64):
            raise NotImplementedError("grid dtype_s must be int64")
    else:  # :593-602
        sp.dtype_s = g("dtype_s", np.float32)
        if g("irrelevant_features", False):
            assert "relevant_indices" in config, \
                "Please provide dimensions of state space relevant to rewards."
        if "relevant_indices" not in config:
            config["relevant_indices"] = range(sp.state_space_dim)
        sp.relevant_indices = [int(i) for i in config["relevant_indices"]]
    sp.dtype_o = g("dtype_o", np.uint8 if sp.image_representations else sp.dtype_s)
    if "init_state_dist" in config and "relevant_init_state_dist" not in config:
        config["relevant_init_state_dist"] = config["init_state_dist"]
    assert sp.sequence_length > 0, \
        'config["sequence_length"] <= 0. Set to: ' + str(sp.sequence_length)
    if kind == "continuous":  # :641-654
        if sp.reward_function == "move_to_a_point":
            assert sp.sequence_length == 1
        if sp.reward_function == "move_along_a_line":
            sp.target_point = None  # (no target: nothing to reach, :1719)
        elif "target_point" in config:
            sp.target_point = np.array(config["target_point"], dtype=sp.dtype_s)
            assert sp.target_point.shape == (len(sp.relevant_indices),), (
                "target_point should have dimensionality = relevant_state_space"
                " dimensionality")
        else:
            sp.target_point = np.zeros((sp.state_space_dim,))
        sp.state_space_max = float(g("state_space_max", np.inf))
        sp.action_space_max = float(g("action_space_max", np.inf))
        if "terminal_states" in config:
            if callable(config["terminal_states"]):
                raise NotImplementedError("callable terminal_states")
            sp.terminal_centres = [list(c) for c in config["terminal_states"]]
            sp.term_state_edge = float(config["term_state_edge"])
            for i, c in enumerate(sp.terminal_centres):
                assert len(c) == len(sp.relevant_indices), (
                    "Specified terminal state centres should have "
                    "dimensionality = number of relevant_indices. That was not"
                    " the case for centre no.: " + str(i))
    return sp
