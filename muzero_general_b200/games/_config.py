"""Shared ``MuZeroConfig`` attribute bag.

The reference has one ``MuZeroConfig`` class per game file (e.g. ``games/cartpole.py:11-128``)
and reads it everywhere as ``self.config.X``; overrides arrive as a dict validated with
``hasattr`` (``muzero.py:54-65``).  The attribute NAMES are the plug-in contract and are
kept verbatim; each game module here fills in that game's values.  Knobs that only this
implementation knows are read with ``getattr(config, name, default)`` on the consuming
side so stock reference configs load unchanged:

* ``num_parallel_games``  games searched in lockstep per GPU process (default 1)
* ``rng_mode``            "numpy" (reference draw order on legacy per-game streams) or
                          "philox" (counter-based, generated on the device)
* ``test_games_per_report``  evaluation games the test worker plays per weight refresh
                          (``SelfPlay.play_test_games``); absent or 0 = one ``play_game`` as in the reference
* ``test_parallel_games`` slots of the device engine that plays evaluation games (default 4096,
                          never more than the games asked for)
"""
import datetime
import pathlib


class BaseMuZeroConfig:
    # (name, default) - defaults are the CartPole file's values
    _DEFAULTS = dict(
        seed=0, max_num_gpus=None,
        observation_shape=(1, 1, 4), action_space=list(range(2)), players=list(range(1)),
        stacked_observations=0, muzero_player=0, opponent=None,
        num_workers=1, selfplay_on_gpu=False, max_moves=500, num_simulations=50, discount=0.997,
        temperature_threshold=None, root_dirichlet_alpha=0.25, root_exploration_fraction=0.25,
        pb_c_base=19652, pb_c_init=1.25,
        network="fullyconnected", support_size=10,
        downsample=False, blocks=1, channels=2,
        reduced_channels_reward=2, reduced_channels_value=2, reduced_channels_policy=2,
        resnet_fc_reward_layers=[], resnet_fc_value_layers=[], resnet_fc_policy_layers=[],
        encoding_size=8, fc_representation_layers=[], fc_dynamics_layers=[16],
        fc_reward_layers=[16], fc_value_layers=[16], fc_policy_layers=[16],
        save_model=True, training_steps=10000, batch_size=128, checkpoint_interval=10,
        value_loss_weight=1, train_on_gpu=False, optimizer="Adam", weight_decay=1e-4, momentum=0.9,
        lr_init=0.02, lr_decay_rate=0.8, lr_decay_steps=1000,
        replay_buffer_size=500, num_unroll_steps=10, td_steps=50, PER=True, PER_alpha=0.5,
        use_last_model_value=True, reanalyse_on_gpu=False,
        self_play_delay=0, training_delay=0, ratio=1.5,
        # additions of this implementation (optional for stock configs)
        num_parallel_games=1, rng_mode="numpy",
    )
    _NAME = "game"
    _OVERRIDES = {}
    # (fraction of training_steps or absolute step, temperature) pairs, last entry = fallback
    _TEMPERATURE_SCHEDULE = ((0.5, 1.0), (0.75, 0.5), (None, 0.25))
    _TEMPERATURE_ABSOLUTE = False

    def __init__(self):
        import copy
        for k, v in self._DEFAULTS.items():
            setattr(self, k, copy.deepcopy(v))
        for k, v in self._OVERRIDES.items():
            setattr(self, k, copy.deepcopy(v))
        self.results_path = (pathlib.Path(__file__).resolve().parents[2] / "results" / self._NAME
                             / datetime.datetime.now().strftime("%Y-%m-%d--%H-%M-%S"))

    def visit_softmax_temperature_fn(self, trained_steps):
        """Greedier action selection as training progresses (e.g. games/cartpole.py:114-128)."""
        for bound, temperature in self._TEMPERATURE_SCHEDULE:
            if bound is None:
                return temperature
            limit = bound if self._TEMPERATURE_ABSOLUTE else bound * self.training_steps
            if trained_steps < limit:
                return temperature
        return self._TEMPERATURE_SCHEDULE[-1][1]


def apply_overrides(config, overrides):
    """Dict / JSON override with the reference's validation (muzero.py:54-65)."""
    if not overrides:
        return config
    if isinstance(overrides, dict):
        for param, value in overrides.items():
            if hasattr(config, param):
                setattr(config, param, value)
            else:
                raise AttributeError(
                    f"{config.__class__.__name__} has no attribute '{param}'. "
                    "Check the config file for the complete list of parameters.")
        return config
    return overrides  # a ready-made config object replaces the default one
