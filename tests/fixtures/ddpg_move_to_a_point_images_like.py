"""A small continuous experiment file with image observations in the
reference's format (cf. its experiments/ddpg_move_to_a_point_time_unit.py
with image_representations on): cells differ in the target and in the size
of the state space, i.e. in what the images show."""
from ray import tune
from collections import OrderedDict

var_env_configs = OrderedDict(
    {
        "state_space_dim": [2],
        "action_space_dim": [2],
        "target_point": [[0, 0], [2.5, -1.5]],
        "target_radius": [0.5],
        "state_space_max": [5, 10],
        "action_space_max": [1],
        "time_unit": [1.0],
    }
)

var_configs = OrderedDict({"env": var_env_configs})

env_config = {
    "env": "RLToy-v0",
    "horizon": 100,
    "env_config": {
        "seed": 0,
        "state_space_type": "continuous",
        "action_space_type": "continuous",
        "inertia": 1,
        "reward_scale": 1.0,
        "reward_function": "move_to_a_point",
        "image_representations": True,
        "image_width": 64,
        "image_height": 48,
    },
}

algorithm = "DDPG"
