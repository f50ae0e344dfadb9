"""A small grid-world experiment file with image observations in the
reference's format (the keys of its grid_image_representations_example):
cells differ in the grid's shape and target, i.e. in what the images show."""
from ray import tune
from collections import OrderedDict

var_env_configs = OrderedDict(
    {
        "grid_shape": [(8, 8), (5, 7)],
        "target_point": [[3, 3], [1, 4]],
        "make_denser": [True],
    }
)

var_configs = OrderedDict({"env": var_env_configs})

env_config = {
    "env": "RLToy-v0",
    "horizon": 50,
    "env_config": {
        "seed": 0,
        "state_space_type": "grid",
        "reward_function": "move_to_a_point",
        "delay": 0,
        "sequence_length": 1,
        "reward_scale": 1.0,
        "terminal_states": [[4, 4]],
        "image_representations": True,
    },
}

algorithm = "DQN"
