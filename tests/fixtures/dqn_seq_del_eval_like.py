"""A small discrete experiment file in the reference's format with the
evaluation settings of its DQN experiment files (cf. its
experiments/dqn_seq_del.py): `eval_config` switches exploration and the
env's noises off for the evaluation episodes."""
from ray import tune
from collections import OrderedDict

num_seeds = 2

var_env_configs = OrderedDict(
    {
        "state_space_size": [8],
        "action_space_size": [8],
        "delay": [0, 1],
        "sequence_length": [1, 2],
        "reward_density": [0.25],
        "make_denser": [False],
        "terminal_state_density": [0.25],
        "transition_noise": [0, 0.1],
        "reward_noise": [0, 0.5],
        "dummy_seed": [i for i in range(num_seeds)],
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
        "reward_every_n_steps": True,
    },
}

algorithm = "DQN"
agent_config = {"lr": tune.grid_search([1e-2, 1e-4])}
model_config = {}

eval_config = {
    "evaluation_interval": 1,  # every training iteration
    "evaluation_config": {
        "explore": False,
        "exploration_fraction": 0,
        "exploration_final_eps": 0,
        "evaluation_num_episodes": 10,
        "horizon": 100,
        "env_config": {
            "dummy_eval": True,  # the reference's callbacks tell evaluation episodes by it
            "transition_noise": 0
            if "state_space_type" in env_config["env_config"]
            and env_config["env_config"]["state_space_type"] == "discrete"
            else tune.function(lambda a: a.normal(0, 0)),
            "reward_noise": tune.function(lambda a: a.normal(0, 0)),
            "action_loss_weight": 0.0,
        },
    },
}
