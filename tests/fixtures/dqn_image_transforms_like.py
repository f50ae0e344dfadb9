"""A small discrete experiment file with image observations in the
reference's format (cf. its experiments/dqn_image_representations_*.py):
cells differ in the image transforms and their quantisation."""
from ray import tune
from collections import OrderedDict

var_env_configs = OrderedDict(
    {
        "state_space_size": [8],
        "action_space_size": [8],
        "delay": [0],
        "sequence_length": [1],
        "reward_density": [0.25],
        "make_denser": [False],
        "terminal_state_density": [0.25],
        "transition_noise": [0],
        "reward_noise": [0],
        "image_transforms": ["none", "shift", "scale", "rotate", "flip",
                             "shift,scale,rotate,flip"],
        "image_sh_quant": [2],
        "image_ro_quant": [10],
        "image_width": [100],
        "image_height": [100],
    }
)

var_configs = OrderedDict({"env": var_env_configs})

env_config = {
    "env": "RLToy-v0",
    "horizon": 100,
    "env_config": {
        "seed": 0,
        "state_space_type": "discrete",
        "action_space_type": "discrete",
        "generate_random_mdp": True,
        "repeats_in_sequences": False,
        "reward_scale": 1.0,
        "completely_connected": True,
        "image_representations": True,
        "image_scale_range": (0.5, 1.5),
    },
}

algorithm = "DQN"
