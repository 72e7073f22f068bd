"""Drop-in self-play surface of the reference (``self_play.py``), backed by libmzb200.so.

Same class names, method names, argument meaning and output format as the reference:

* ``SelfPlay(initial_checkpoint, Game, config, seed)`` with ``continuous_self_play``,
  ``play_game``, ``close_game``, ``select_opponent_action`` and the static
  ``select_action``                                              (self_play.py:11-245)
* ``MCTS(config).run(model, observation, legal_actions, to_play, add_exploration_noise)``
  returning ``(root Node, {"max_tree_depth", "root_predicted_value"})``   (self_play.py:249-361)
* ``Node`` with ``children / visit_count / value_sum / prior / reward / hidden_state /
  to_play / expanded() / value()``                               (self_play.py:433-476)
* ``GameHistory`` with the exact attribute set ``ReplayBuffer.save_game`` and
  ``Trainer`` consume (self_play.py:479-550; replay_buffer.py:33-65,85-111,230-303)
* ``MinMaxStats``                                                (self_play.py:553-570)

What changes is HOW a move is computed: every search is a call into the CUDA library, and
``config.num_parallel_games`` games can be searched in lockstep by one process
(``SelfPlay.play_games`` / ``self_play_stream``).  With one game and ``rng_mode="numpy"`` the
draw order on the legacy global ``numpy.random`` stream is the reference's: Dirichlet noise,
then the first simulation's uniform pick, then the action sample.
"""
from __future__ import annotations

import time
from collections import deque

import numpy

from .engine import DeviceSelfPlayLoop, SearchEngine, parse_staged_game


# ----------------------------------------------------------------------------------------
# remote-or-local call helpers: the reference talks to Ray actors (self_play.py:32-37);
# plain objects with the same methods work too.
# ----------------------------------------------------------------------------------------
def _call(obj, method, *args):
    fn = getattr(obj, method)
    if hasattr(fn, "remote"):
        import ray
        return ray.get(fn.remote(*args))
    return fn(*args)


def _fire(obj, method, *args):
    fn = getattr(obj, method)
    if hasattr(fn, "remote"):
        return fn.remote(*args)
    return fn(*args)


# ----------------------------------------------------------------------------------------
# model facade
# ----------------------------------------------------------------------------------------
class DeviceModel:
    """Stands where ``models.MuZeroNetwork(config)`` stood in ``SelfPlay`` (self_play.py:25-29).

    Holds the CUDA search engine; ``set_weights`` / ``get_weights`` keep the reference's
    state_dict format (models.py:69-73).
    """

    def __init__(self, config, max_games=1, device=0, seed=None, num_simulations=None):
        self.config = config
        # a single-game model also serves MCTS.run(override_root_with=...) (diagnose_model.py:61-72): the continued
        # search adds num_simulations expansions to an imported subtree of up to num_simulations expansions
        n = int(config.num_simulations if num_simulations is None else num_simulations)
        self.engine = SearchEngine(config, max_games=max_games, device=device, seed=seed,
                                   num_simulations=num_simulations, extra_expansions=n + 1 if max_games == 1 else 0)
        self._weights = None

    def set_weights(self, weights):
        self.engine.load_weights(weights)
        self._weights = weights

    def get_weights(self):
        return self._weights

    def eval(self):
        return self

    def to(self, device):
        return self

    def initial_inference(self, observation):
        """[B,C',H,W] -> (value_logits, reward_logits, policy_logits, hidden) as torch tensors."""
        import torch
        obs = numpy.asarray(observation.cpu() if hasattr(observation, "cpu") else observation, dtype=numpy.float32)
        r = self.engine.initial_inference(obs)
        return (torch.from_numpy(r["value_logits"]), torch.from_numpy(r["reward_logits"]),
                torch.from_numpy(r["policy_logits"]), torch.from_numpy(r["hidden"]))

    def recurrent_inference(self, encoded_state, action):
        import torch
        h = numpy.asarray(encoded_state.cpu() if hasattr(encoded_state, "cpu") else encoded_state, dtype=numpy.float32)
        a = numpy.asarray(action.cpu() if hasattr(action, "cpu") else action).reshape(-1)
        r = self.engine.recurrent_inference(h.reshape(h.shape[0], -1), a)
        return (torch.from_numpy(r["value_logits"]), torch.from_numpy(r["reward_logits"]),
                torch.from_numpy(r["policy_logits"]), torch.from_numpy(r["hidden"]))


# ----------------------------------------------------------------------------------------
# tree view
# ----------------------------------------------------------------------------------------
class Node:
    """Read-only mirror of the reference ``Node`` (self_play.py:433-449) built from the device tree."""

    def __init__(self, prior):
        self.visit_count = 0
        self.to_play = -1
        self.prior = prior
        self.value_sum = 0
        self.children = {}
        self.hidden_state = None
        self.reward = 0

    def expanded(self):
        return len(self.children) > 0

    def value(self):
        if self.visit_count == 0:
            return 0
        return self.value_sum / self.visit_count

    def expand(self, actions, to_play, reward, policy_logits, hidden_state):
        """Fill the node from a network output (self_play.py:451-465) - host side, for callers that build a root by
        hand before ``MCTS.run(..., override_root_with=root)`` (diagnose_model.py:54-69)."""
        import torch
        self.to_play = to_play
        self.reward = reward
        self.hidden_state = hidden_state
        policy_values = torch.softmax(torch.tensor([policy_logits[0][a] for a in actions]), dim=0).tolist()
        for i, action in enumerate(actions):
            self.children[action] = Node(policy_values[i])

    def add_exploration_noise(self, dirichlet_alpha, exploration_fraction):
        """self_play.py:467-476."""
        actions = list(self.children.keys())
        noise = numpy.random.dirichlet([dirichlet_alpha] * len(actions))
        frac = exploration_fraction
        for a, n in zip(actions, noise):
            self.children[a].prior = self.children[a].prior * (1 - frac) + n * frac


def _flatten_subtree(root, A, hidden_elems):
    """``Node`` graph -> the struct-of-arrays tree ``mz_import_tree`` takes: expansion 0 = ``root``, expanded
    children numbered breadth first, child slots ``[e*A, e*A+A)`` by action id."""
    nodes, order = [root], {id(root): 0}
    i = 0
    while i < len(nodes):
        for a in range(A):
            ch = nodes[i].children.get(a)
            if ch is not None and ch.expanded():
                order[id(ch)] = len(nodes)
                nodes.append(ch)
        i += 1
    K = len(nodes)
    t = dict(n_expansions=K, child_visit=numpy.zeros(K * A, numpy.int32), child_value_sum=numpy.zeros(K * A),
             child_reward=numpy.zeros(K * A, numpy.float32), child_prior=numpy.zeros(K * A),
             child_expansion=numpy.full(K * A, -1, numpy.int32), hidden=numpy.zeros((K, hidden_elems), numpy.float32),
             root_visit=int(root.visit_count), root_value_sum=float(root.value_sum), root_reward=float(root.reward))
    for e, node in enumerate(nodes):
        assert set(node.children) == set(range(A)), "override_root_with: an expanded non-root node has every action as a child"
        t["hidden"][e] = numpy.asarray(node.hidden_state, dtype=numpy.float32).ravel()
        for a, ch in node.children.items():
            s = e * A + a
            t["child_visit"][s] = ch.visit_count
            t["child_value_sum"][s] = ch.value_sum
            t["child_prior"][s] = ch.prior
            if ch.expanded():
                t["child_reward"][s] = ch.reward
                t["child_expansion"][s] = order[id(ch)]
    return t


def _node_graph(tree, legal_actions, to_play, num_players, A):
    """Rebuild the ``Node`` graph of one game from ``SearchEngine.export_tree``."""
    root = Node(0)
    root.visit_count = tree["root_visit"]
    root.value_sum = tree["root_value_sum"]
    root.to_play = to_play
    root.reward = tree.get("root_reward", -0.0)
    hidden = tree.get("hidden")
    if hidden is not None:
        root.hidden_state = hidden[0]
    stack = [(root, 0, to_play)]
    while stack:
        node, e, tp = stack.pop()
        actions = legal_actions if e == 0 else range(A)
        nxt = (tp + 1) % num_players
        for a in actions:
            s = e * A + a
            child = Node(float(tree["child_prior"][s]))
            child.visit_count = int(tree["child_visit"][s])
            child.value_sum = float(tree["child_value_sum"][s])
            node.children[a] = child
            ce = int(tree["child_expansion"][s])
            if ce >= 0:
                child.reward = float(tree["child_reward"][s])
                child.to_play = nxt
                if hidden is not None:
                    child.hidden_state = hidden[ce]
                stack.append((child, ce, nxt))
    return root


class MCTS:
    """``MCTS(config).run`` for ONE game through the batched engine (self_play.py:249-361)."""

    def __init__(self, config):
        self.config = config

    def run(self, model, observation, legal_actions, to_play, add_exploration_noise, override_root_with=None):
        config = self.config
        if override_root_with:
            return self._continue(model, legal_actions, to_play, add_exploration_noise, override_root_with)
        assert legal_actions, f"Legal actions should not be an empty array. Got {legal_actions}."
        assert set(legal_actions).issubset(set(config.action_space)), \
            "Legal actions should be a subset of the action space."
        assert list(legal_actions) == sorted(legal_actions), "legal_actions must be ascending"
        engine = model.engine
        A = engine.A
        mask = numpy.zeros((1, A), numpy.uint8)
        mask[0, list(legal_actions)] = 1
        noise = None
        if add_exploration_noise:
            draw = numpy.random.dirichlet([config.root_dirichlet_alpha] * len(legal_actions))   # self_play.py:473
            noise = numpy.zeros((1, A))
            noise[0, list(legal_actions)] = draw
        # first simulation: every root child scores exactly 0 -> uniform pick (self_play.py:371)
        first = list(legal_actions).index(numpy.random.choice(list(legal_actions)))
        obs = numpy.asarray(observation, dtype=numpy.float32)[None]
        out = engine.search(obs=obs, legal_mask=mask, to_play=numpy.array([to_play], numpy.int32),
                            add_exploration_noise=add_exploration_noise, noise=noise,
                            first_index=numpy.array([first], numpy.int32), keep_tree=True)
        tree = engine.export_tree(0, with_hidden=True)
        root = _node_graph(tree, list(legal_actions), to_play, len(config.players), A)
        return root, {"max_tree_depth": int(out.max_tree_depth[0]),
                      "root_predicted_value": float(out.root_predicted_value[0])}


# ----------------------------------------------------------------------------------------
# output format
# ----------------------------------------------------------------------------------------
def _mcts_continue(self, model, legal_actions, to_play, add_exploration_noise, node):
    """``MCTS.run(..., override_root_with=node)`` (self_play.py:275-277; diagnose_model.py:61-72): ``node`` - an expanded
    node of an earlier search, typically ``root.children[action]`` - becomes the root, ``num_simulations`` more
    simulations are run on top of what it already holds, with fresh ``MinMaxStats``; ``root_predicted_value`` is None.
    The subtree is uploaded with ``mz_import_tree`` and searched with ``MZ_FLAG_CONTINUE``; a new ``Node`` graph is
    returned (the reference mutates ``node`` in place)."""
    config = self.config
    engine = model.engine
    A = engine.A
    assert node.expanded(), "override_root_with needs an expanded node"
    assert list(legal_actions) == list(range(A)), "a non-root node has the whole action space as children"
    tree = _flatten_subtree(node, A, engine.hidden_elems)
    engine.import_tree(0, tree)
    noise, first = None, None
    if add_exploration_noise:
        noise = numpy.random.dirichlet([config.root_dirichlet_alpha] * A)[None]     # self_play.py:473 on the node's children
    if node.visit_count == 0:
        # an unvisited root: every child scores exactly 0 in the first simulation -> uniform pick (self_play.py:371)
        first = numpy.array([numpy.random.choice(A)], numpy.int32)
    out = engine.search(legal_mask=numpy.ones((1, A), numpy.uint8), to_play=numpy.array([to_play], numpy.int32),
                        add_exploration_noise=add_exploration_noise, noise=noise, first_index=first, keep_tree=True,
                        continue_tree=True, n_games=1)
    new = engine.export_tree(0, with_hidden=True)
    root = _node_graph(new, list(range(A)), to_play, len(config.players), A)
    return root, {"max_tree_depth": int(out.max_tree_depth[0]), "root_predicted_value": None}


MCTS._continue = _mcts_continue


class GameHistory:
    """Same attributes and helpers as the reference's (self_play.py:479-550)."""

    def __init__(self):
        self.observation_history = []
        self.action_history = []
        self.reward_history = []
        self.to_play_history = []
        self.child_visits = []
        self.root_values = []
        self.reanalysed_predicted_root_values = None
        # For PER
        self.priorities = None
        self.game_priority = None

    def store_search_statistics(self, root, action_space):
        if root is not None:
            total = sum(child.visit_count for child in root.children.values())
            self.child_visits.append(
                [root.children[a].visit_count / total if a in root.children else 0 for a in action_space])
            self.root_values.append(root.value())
        else:
            self.root_values.append(None)

    def store_visit_counts(self, visit_counts, legal_mask, root_value, action_space):
        """Batched equivalent of ``store_search_statistics``: one row of the engine's output."""
        total = int(visit_counts.sum())
        self.child_visits.append([int(visit_counts[a]) / total if legal_mask[a] else 0 for a in action_space])
        self.root_values.append(float(root_value))

    def get_stacked_observations(self, index, num_stacked_observations, action_space_size):
        index = index % len(self.observation_history)
        planes = [self.observation_history[index].copy()]
        like = planes[0][0]
        for past in range(index - 1, index - num_stacked_observations - 1, -1):
            if past >= 0:
                planes.append(self.observation_history[past])
                planes.append([numpy.ones_like(like) * self.action_history[past + 1] / action_space_size])
            else:
                planes.append(numpy.zeros_like(self.observation_history[index]))
                planes.append([numpy.zeros_like(like)])
        return numpy.concatenate(planes) if len(planes) > 1 else planes[0]


class MinMaxStats:
    """self_play.py:553-570 (the device keeps the same two doubles per game)."""

    def __init__(self):
        self.maximum = -float("inf")
        self.minimum = float("inf")

    def update(self, value):
        self.maximum = max(self.maximum, value)
        self.minimum = min(self.minimum, value)

    def normalize(self, value):
        if self.maximum > self.minimum:
            return (value - self.minimum) / (self.maximum - self.minimum)
        return value


class PackedGameHistory(GameHistory):
    """A finished game as it left the device (one packed struct-of-arrays block, ``mz_selfplay_drain``), presented
    as a ``GameHistory``.  The reference's list attributes (self_play.py:485-494) are built on first access - a
    consumer that only counts games or forwards them pays nothing per position - and the object pickles as a plain
    ``GameHistory``, so the reference's ReplayBuffer / Trainer / replay_buffer.pkl see the usual type."""

    _LISTS = ("observation_history", "action_history", "reward_history", "to_play_history", "child_visits", "root_values")

    def __init__(self, packed, obs_shape, obs_dtype, reward_type, with_priorities=False):
        # deliberately NOT calling GameHistory.__init__: the six lists stay absent until asked for
        self.__dict__["_packed"] = (packed, tuple(obs_shape), obs_dtype, reward_type)
        self.reanalysed_predicted_root_values = None
        self.priorities = None
        self.game_priority = None
        if with_priorities:
            # computed by the packing warp on the device (replay_buffer.py:39-51): save_game keeps them as they are
            self.priorities = packed["priority"].copy()
            self.game_priority = numpy.max(self.priorities)

    def __len__(self):
        return int(self._packed[0]["length"])

    @property
    def game_id(self):
        return int(self._packed[0]["game_id"])

    def __getattr__(self, name):
        if name in PackedGameHistory._LISTS and "_packed" in self.__dict__:
            self._materialise()
            return self.__dict__[name]
        raise AttributeError(name)

    def _materialise(self):
        g, shape, dtype, reward_type = self._packed
        T = int(g["length"])
        obs = g["obs"].reshape((T + 1,) + shape).astype(dtype)
        d = self.__dict__
        d["observation_history"] = list(obs)
        d["action_history"] = [0] + list(g["action"].astype(numpy.int64))
        d["reward_history"] = [0] + [reward_type(r) for r in g["reward"].tolist()]
        d["to_play_history"] = [int(g["first_to_play"])] + g["to_play"].tolist()
        visits = g["visits"]
        searched = visits.sum(1) > 0
        if searched.all():
            d["child_visits"] = (visits / visits.sum(1, keepdims=True)).tolist()
            d["root_values"] = g["root_value"].tolist()
        else:
            # evaluation games: the opponent's moves carry no search statistics, like store_search_statistics(None, ...)
            # (self_play.py:175,496-511): no child_visits row, root value None
            visits = visits[searched]
            d["child_visits"] = (visits / visits.sum(1, keepdims=True)).tolist()
            d["root_values"] = [v if ok else None for v, ok in zip(g["root_value"].tolist(), searched.tolist())]

    def __reduce__(self):
        self._materialise()
        state = {k: v for k, v in self.__dict__.items() if k != "_packed"}
        return (object.__new__, (GameHistory,), state)      # unpickles as a plain GameHistory, no helper of ours needed


def register_as_reference_module():
    """Make pickles of ``GameHistory`` interchangeable with the reference's replay_buffer.pkl
    (muzero.py:338-346,444-446): the class is published under the module name ``self_play``."""
    import sys
    import types
    mod = sys.modules.get("self_play")
    if mod is None:
        mod = types.ModuleType("self_play")
        sys.modules["self_play"] = mod
    for cls in (GameHistory, MinMaxStats, Node, MCTS, SelfPlay):
        setattr(mod, cls.__name__, cls)
    GameHistory.__module__ = "self_play"


# ----------------------------------------------------------------------------------------
# the actor
# ----------------------------------------------------------------------------------------
class SelfPlay:
    """Plays games and saves them to the replay buffer (self_play.py:11-245)."""

    def __init__(self, initial_checkpoint, Game, config, seed, device=0, first_game_id=0, game_id_stride=None):
        self.config = config
        self.device = device
        self.first_game_id = int(first_game_id)      # rank * num_parallel_games in a multi-GPU job
        # a slot's next game takes (current id + stride): world_size * num_parallel_games keeps ids unique over ranks
        self.game_id_stride = int(game_id_stride or getattr(config, "num_parallel_games", 1) or 1)
        self.Game = Game
        self.seed = seed
        self.num_parallel_games = int(getattr(config, "num_parallel_games", 1) or 1)
        self.rng_mode = getattr(config, "rng_mode", "numpy")
        self.game = Game(seed)

        # Fix random generator seed (self_play.py:22-23)
        numpy.random.seed(seed)

        self.model = DeviceModel(config, max_games=self.num_parallel_games, device=device, seed=seed)
        self.model.set_weights(initial_checkpoint["weights"])
        self._device_loop = None      # device-resident variant of the same (play_moves)
        self._batched = None          # persistent lockstep batch: environments, RNG streams and game ids carry
        self._stream = None           # across play_games calls (its generator)
        self.played_games = 0
        self.played_steps = 0
        self._test_model = None       # evaluation games on the device (play_test_games): own engine, own game ids
        self._next_test_game_id = 0
        self.last_test_searches = 0   # positions the last device evaluation searched, games dropped beyond the ids included

    # ------------------------------------------------------------------ reference loop
    def continuous_self_play(self, shared_storage, replay_buffer, test_mode=False):
        cfg = self.config
        while (_call(shared_storage, "get_info", "training_step") < cfg.training_steps
               and not _call(shared_storage, "get_info", "terminate")):
            self.model.set_weights(_call(shared_storage, "get_info", "weights"))
            if not test_mode:
                temperature = cfg.visit_softmax_temperature_fn(
                    trained_steps=_call(shared_storage, "get_info", "training_step"))
                if self.num_parallel_games > 1:
                    # the lockstep batch advances between two weight refreshes; every finished game goes to the buffer
                    if self.loop_path == "device":
                        games = self.play_moves(int(getattr(cfg, "moves_per_weight_refresh", 8)), temperature,
                                                cfg.temperature_threshold)
                    else:
                        games = self.play_games(self.num_parallel_games, temperature, cfg.temperature_threshold)
                    for game_history in games:
                        _fire(replay_buffer, "save_game", game_history, shared_storage)
                else:
                    game_history = self.play_game(temperature, cfg.temperature_threshold, False, "self", 0)
                    _fire(replay_buffer, "save_game", game_history, shared_storage)
            elif int(getattr(cfg, "test_games_per_report", 0) or 0):
                # a batch of evaluation games per weight refresh: the reference's keys averaged over the games
                _, summary = self.play_test_games(int(cfg.test_games_per_report))
                _fire(shared_storage, "set_info", {k: summary[k] for k in ("episode_length", "total_reward", "mean_value")})
                if 1 < len(cfg.players):
                    _fire(shared_storage, "set_info", {k: summary[k] for k in ("muzero_reward", "opponent_reward")})
            else:
                # Take the best action (no exploration) in test mode
                game_history = self.play_game(
                    0, cfg.temperature_threshold, False,
                    "self" if len(cfg.players) == 1 else cfg.opponent, cfg.muzero_player)
                _fire(shared_storage, "set_info", {
                    "episode_length": len(game_history.action_history) - 1,
                    "total_reward": sum(game_history.reward_history),
                    "mean_value": numpy.mean([value for value in game_history.root_values if value]),
                })
                if 1 < len(cfg.players):
                    _fire(shared_storage, "set_info", {
                        "muzero_reward": sum(
                            reward for i, reward in enumerate(game_history.reward_history)
                            if game_history.to_play_history[i - 1] == cfg.muzero_player),
                        "opponent_reward": sum(
                            reward for i, reward in enumerate(game_history.reward_history)
                            if game_history.to_play_history[i - 1] != cfg.muzero_player),
                    })

            # Managing the self-play / training ratio
            if not test_mode and cfg.self_play_delay:
                time.sleep(cfg.self_play_delay)
            if not test_mode and cfg.ratio:
                while (_call(shared_storage, "get_info", "training_step")
                       / max(1, _call(shared_storage, "get_info", "num_played_steps")) < cfg.ratio
                       and _call(shared_storage, "get_info", "training_step") < cfg.training_steps
                       and not _call(shared_storage, "get_info", "terminate")):
                    time.sleep(0.5)
        self.close_game()

    def play_game(self, temperature, temperature_threshold, render, opponent, muzero_player):
        """One game, one search per move (self_play.py:110-183)."""
        cfg = self.config
        game_history = GameHistory()
        observation = self.game.reset()
        game_history.action_history.append(0)
        game_history.observation_history.append(observation)
        game_history.reward_history.append(0)
        game_history.to_play_history.append(self.game.to_play())
        done = False
        if render:
            self.game.render()
        while not done and len(game_history.action_history) <= cfg.max_moves:
            assert len(numpy.array(observation).shape) == 3, \
                f"Observation should be 3 dimensionnal instead of {len(numpy.array(observation).shape)} dimensionnal. Got observation of shape: {numpy.array(observation).shape}"
            assert numpy.array(observation).shape == cfg.observation_shape, \
                f"Observation should match the observation_shape defined in MuZeroConfig. Expected {cfg.observation_shape} but got {numpy.array(observation).shape}."
            stacked_observations = game_history.get_stacked_observations(
                -1, cfg.stacked_observations, len(cfg.action_space))

            # Choose the action
            if opponent == "self" or muzero_player == self.game.to_play():
                root, mcts_info = MCTS(cfg).run(self.model, stacked_observations, self.game.legal_actions(),
                                                self.game.to_play(), True)
                action = self.select_action(
                    root,
                    temperature if not temperature_threshold
                    or len(game_history.action_history) < temperature_threshold else 0)
                if render:
                    print(f'Tree depth: {mcts_info["max_tree_depth"]}')
                    print(f"Root value for player {self.game.to_play()}: {root.value():.2f}")
            else:
                action, root = self.select_opponent_action(opponent, stacked_observations)

            observation, reward, done = self.game.step(action)
            if render:
                print(f"Played action: {self.game.action_to_string(action)}")
                self.game.render()
            game_history.store_search_statistics(root, cfg.action_space)

            # Next batch
            game_history.action_history.append(action)
            game_history.observation_history.append(observation)
            game_history.reward_history.append(reward)
            game_history.to_play_history.append(self.game.to_play())
        self.played_games += 1
        self.played_steps += len(game_history.action_history) - 1
        return game_history

    def close_game(self):
        self.game.close()

    def select_opponent_action(self, opponent, stacked_observations):
        """Opponent move for evaluation games (self_play.py:188-220)."""
        if opponent == "human":
            root, mcts_info = MCTS(self.config).run(self.model, stacked_observations, self.game.legal_actions(),
                                                    self.game.to_play(), True)
            print(f'Tree depth: {mcts_info["max_tree_depth"]}')
            print(f"Root value for player {self.game.to_play()}: {root.value():.2f}")
            print(f"Player {self.game.to_play()} turn. MuZero suggests "
                  f"{self.game.action_to_string(self.select_action(root, 0))}")
            return self.game.human_to_action(), root
        elif opponent == "expert":
            return self.game.expert_agent(), None
        elif opponent == "random":
            assert self.game.legal_actions(), \
                f"Legal actions should not be an empty array. Got {self.game.legal_actions()}."
            assert set(self.game.legal_actions()).issubset(set(self.config.action_space)), \
                "Legal actions should be a subset of the action space."
            return numpy.random.choice(self.game.legal_actions()), None
        raise NotImplementedError(
            'Wrong argument: "opponent" argument should be "self", "human", "expert" or "random"')

    # ------------------------------------------------------------------ evaluation games
    def play_test_games(self, num_games, opponent=None, muzero_player=None, first_game_id=None):
        """``num_games`` evaluation games, the batched ``MuZero.test`` (muzero.py:369-424) and test worker
        (self_play.py:54-90): greedy moves with root noise, as ``play_game(0, 0, False, opponent, muzero_player)``.

        ``opponent`` / ``muzero_player`` = None take ``config.opponent`` / ``config.muzero_player`` (an explicit 0 is
        kept); one-player games always play "self"; "human" is not supported.  Returns ``(games, summary)``: the games
        (``PackedGames`` from the device loop, else a list of ``GameHistory``) and ``evaluation_summary`` of them.

        With a device-resident environment (``loop_path == "device"``) the games run in ``mz_selfplay_*`` on an engine of
        their own with ``min(num_games, config.test_parallel_games or 4096)`` slots, loaded with the worker's current
        weights; the self-play batch in flight is not touched.  Exactly the global game ids ``[first_game_id,
        first_game_id + num_games)`` are returned (games the slots start beyond them are dropped), so the result does not
        depend on the number of slots; ``first_game_id`` = None continues after the previous call.  Otherwise
        ``play_game`` is called ``num_games`` times."""
        cfg = self.config
        opponent, muzero_player = resolve_opponent(cfg, opponent, muzero_player)
        num_games = int(num_games)
        first = self._next_test_game_id if first_game_id is None else int(first_game_id)
        if self._device_env_name():
            games = self._device_test_games(num_games, opponent, muzero_player, first)
        else:
            games = [self.play_game(0, 0, False, opponent, muzero_player) for _ in range(num_games)]
        self._next_test_game_id = first + num_games
        return games, evaluation_summary(games, len(cfg.players), muzero_player)

    def _device_test_games(self, num_games, opponent, muzero_player, first):
        cfg, Game = self.config, self.Game
        B = max(1, min(num_games, int(getattr(cfg, "test_parallel_games", 0) or 4096)))
        if self._test_model is None or self._test_model.engine.max_games != B:
            if self._test_model is not None:
                self._test_model.engine.close()
            self._test_model = DeviceModel(cfg, max_games=B, device=self.device, seed=self.seed)
        self._test_model.set_weights(self.model.get_weights())
        vec = getattr(Game, "VECTOR", None)
        loop = DeviceSelfPlayLoop(self._test_model.engine, Game.DEVICE_ENV, cfg.max_moves,
                                  reward_scale=getattr(vec, "REWARD_SCALE", 1), first_game_id=first, game_id_stride=B,
                                  opponent=opponent, muzero_player=muzero_player)
        out = PackedGames(tuple(cfg.observation_shape), getattr(vec, "OBS_DTYPE", numpy.float32),
                          int if vec is not None else float)
        end = first + num_games
        searches = 0
        while len(out) < num_games:
            # one batched move per call: the evaluation stops right after the last wanted game ends (a move costs a
            # search of the whole batch, the host round trip is small beside it)
            loop.moves(1, 0.0)
            searches += 1
            buf, index = loop.drain()
            if len(index):
                ids = numpy.frombuffer(buf, numpy.int64)[(index[:, 0] // 8).astype(numpy.int64)]
                out.add(buf, index[ids < end])
        self.played_games += len(out)
        self.played_steps += out.total_moves
        self.last_test_searches = searches * B
        return out

    @staticmethod
    def select_action(node, temperature):
        """Visit-count sampling (self_play.py:222-245)."""
        visit_counts = numpy.array([child.visit_count for child in node.children.values()], dtype="int32")
        actions = [action for action in node.children.keys()]
        return _sample_action(actions, visit_counts, temperature, numpy.random)

    # ------------------------------------------------------------------ batched play
    def play_games(self, num_games, temperature, temperature_threshold=None, max_total_moves=None):
        """The next ``num_games`` finished games of the worker's lockstep batch (``num_parallel_games`` games in flight).

        The batch is PERSISTENT: games still in flight when the quota is reached keep their state and finish in a
        later call (long episodes are not dropped), every game gets a fresh global id / RNG stream, and a weight
        refresh between calls (``continuous_self_play``) simply applies to the remaining moves - like a reference
        actor that reloads weights between games.  ``max_total_moves`` bounds the env-steps of THIS call."""
        stream = self.self_play_stream(temperature, temperature_threshold)
        start = self._batched.env_steps
        out = []
        while len(out) < num_games:
            out.append(next(stream))
            if max_total_moves is not None and self._batched.env_steps - start >= max_total_moves:
                break
        return out

    def self_play_stream(self, temperature, temperature_threshold=None):
        """Generator over finished ``GameHistory`` objects; B games advance one move per iteration."""
        if self._batched is None:
            self._batched = BatchedSelfPlay(self, temperature, temperature_threshold, self.first_game_id)
            self._stream = self._batched.run()
        else:
            self._batched.temperature = temperature
            self._batched.temperature_threshold = temperature_threshold
        return self._stream

    def reset_stream(self):
        """Drop the games in flight (e.g. after changing ``config`` fields the batch was built from)."""
        self._batched = None
        self._stream = None
        self._device_loop = None

    # ------------------------------------------------------------------ whole-batch moves
    def _device_env_name(self):
        """Name of the device-resident environment for this worker, or None (host environments)."""
        cfg = self.config
        name = getattr(self.Game, "DEVICE_ENV", None)
        if (name is None or self.rng_mode != "philox" or cfg.stacked_observations
                or not getattr(cfg, "device_envs", True)):
            return None
        return name

    @property
    def loop_path(self):
        """"device": environments, sampling and records on the GPU (mz_selfplay_*); "host": numpy environments."""
        return "device" if self._device_env_name() else "host"

    @property
    def env_steps(self):
        """Moves played by the lockstep batch so far (finished games or not)."""
        if getattr(self, "_device_loop", None) is not None:
            return int(self._device_loop.loop.stats.env_steps)
        return self._batched.env_steps if self._batched is not None else 0

    def play_moves(self, n_moves, temperature, temperature_threshold=None):
        """Advance every game of the lockstep batch by ``n_moves`` moves; returns the games that finished.

        With ``rng_mode="philox"`` and a game that has a device-resident environment (CartPole, TicTacToe, Connect4)
        the whole loop - observation, search, visit-count sampling, environment step, history records - runs on the
        GPU (``mz_selfplay_moves``) and only finished games cross to the host, as ``PackedGameHistory`` objects.
        Otherwise the host loop (``BatchedSelfPlay.move``) is used."""
        if self._device_env_name():
            if getattr(self, "_device_loop", None) is None:
                self._device_loop = DeviceBatchedSelfPlay(self, temperature_threshold)
            games = self._device_loop.moves(n_moves, temperature)
            self.played_games += len(games)
            self.played_steps += games.total_moves
            return games
        self.self_play_stream(temperature, temperature_threshold)
        out = []
        for _ in range(n_moves):
            out.extend(self._batched.move())
        return out

    def close(self):
        self.model.engine.close()


def resolve_opponent(config, opponent=None, muzero_player=None):
    """(opponent, muzero_player) of an evaluation: None takes the config's value (an explicit 0 is kept, where
    muzero.py:390's ``if muzero_player`` would replace it); a one-player game plays "self" (self_play.py:60)."""
    if opponent == "human":
        raise ValueError('opponent "human" is interactive: use play_game for it')
    opponent = config.opponent if opponent is None else opponent
    muzero_player = int(config.muzero_player if muzero_player is None else muzero_player)
    if len(config.players) == 1:
        return "self", muzero_player
    if opponent not in ("self", "expert", "random"):
        raise ValueError(f'opponent must be "self", "expert" or "random", got {opponent!r}')
    return opponent, muzero_player


def evaluation_summary(games, num_players, muzero_player):
    """Test-worker statistics (self_play.py:67-90) of every game, averaged over the games, plus ``MuZero.test``'s
    ``result`` (muzero.py:411-424).  ``games``: ``GameHistory`` objects or ``PackedGames`` (read from the packed reward /
    to_play / root-value arrays, nothing materialised).  Per game, as the reference computes it:
      episode_length = moves; total_reward = sum of rewards; mean_value = mean of the root values that are truthy
      (neither None nor 0.0; NaN for a game without one); muzero_reward / opponent_reward = rewards of the moves played by
      muzero_player / the other side.
    A game whose mean_value is NaN is left out of that average.  Two-player games also get the keys muzero_reward,
    opponent_reward and wins / draws / losses (muzero_reward above / equal to / below opponent_reward)."""
    rows = []                 # per game: length, total reward, mean value, muzero reward, opponent reward
    if isinstance(games, PackedGames):
        for g in games.blocks():
            rewards = g["reward"].astype(numpy.float64)
            mover = numpy.concatenate(([g["first_to_play"]], g["to_play"][:-1]))
            root = g["root_value"]
            values = root[~numpy.isnan(root) & (root != 0)]
            rows.append((g["length"], float(rewards.sum()), float(values.mean()) if values.size else numpy.nan,
                         float(rewards[mover == muzero_player].sum()), float(rewards[mover != muzero_player].sum())))
    else:
        for h in games:
            rh, tp = h.reward_history, h.to_play_history
            values = [value for value in h.root_values if value]
            with numpy.errstate(invalid="ignore", divide="ignore"):
                mean_value = float(numpy.mean(values)) if values else numpy.nan
            rows.append((len(h.action_history) - 1, sum(rh), mean_value,
                         sum(reward for i, reward in enumerate(rh) if tp[i - 1] == muzero_player),
                         sum(reward for i, reward in enumerate(rh) if tp[i - 1] != muzero_player)))
    n = len(rows)
    col = (lambda k: numpy.array([r[k] for r in rows], numpy.float64)) if n else (lambda k: numpy.zeros(0))
    mean = lambda a: float(numpy.mean(a)) if a.size else numpy.nan
    mv = col(2)
    mv = mv[~numpy.isnan(mv)]
    out = dict(num_games=n, episode_length=mean(col(0)), total_reward=mean(col(1)), mean_value=mean(mv))
    if num_players > 1:
        mine, theirs = col(3), col(4)
        out.update(muzero_reward=mean(mine), opponent_reward=mean(theirs), wins=int((mine > theirs).sum()),
                   draws=int((mine == theirs).sum()), losses=int((mine < theirs).sum()), result=mean(mine))
    else:
        out["result"] = out["total_reward"]
    return out


def _sample_action(actions, visit_counts, temperature, rng):
    if temperature == 0:
        return actions[numpy.argmax(visit_counts)]
    if temperature == float("inf"):
        return rng.choice(actions)
    # See paper appendix Data Generation
    dist = visit_counts ** (1 / temperature)
    dist = dist / sum(dist)
    return rng.choice(actions, p=dist)


class _ObjectVector:
    """Adapter giving ``num_games`` ordinary ``Game`` objects the ``VectorGame`` interface."""

    def __init__(self, Game, num_games, seed, A):
        self.games = [Game(seed + g) for g in range(num_games)]
        self.num_games = num_games
        self.A = A
        self._obs = [None] * num_games

    def reset(self, which=None):
        idx = range(self.num_games) if which is None else numpy.nonzero(which)[0]
        for g in idx:
            self._obs[g] = numpy.asarray(self.games[g].reset())
        return self._obs

    def observations(self):
        return self._obs

    def step(self, actions):
        rewards, dones = [], []
        for g, game in enumerate(self.games):
            o, r, d = game.step(actions[g])
            self._obs[g] = numpy.asarray(o)
            rewards.append(r)
            dones.append(d)
        return self._obs, rewards, numpy.array(dones, dtype=bool)

    def legal_mask(self):
        m = numpy.zeros((self.num_games, self.A), numpy.uint8)
        for g, game in enumerate(self.games):
            m[g, game.legal_actions()] = 1
        return m

    def to_play(self):
        return numpy.array([game.to_play() for game in self.games], dtype=numpy.int32)


class DeviceBatchedSelfPlay:
    """Lockstep self-play with the environments on the GPU (SURVEY.md 8f-1): per call ONE ``mz_selfplay_moves`` for
    ``n_moves`` moves of the whole batch, then one read of the packed finished games.  Slot g plays the global games
    ``first_game_id + g + k*B``; every random draw is a Philox stream keyed by (seed, global game id, move), so a
    game's history is independent of the batch size and of the number of ranks."""

    def __init__(self, worker, temperature_threshold=None):
        cfg = worker.config
        Game = worker.Game
        vec = getattr(Game, "VECTOR", None)
        self.obs_shape = tuple(cfg.observation_shape)
        self.obs_dtype = getattr(vec, "OBS_DTYPE", numpy.float32)
        self.reward_type = int if vec is not None else float
        self.loop = DeviceSelfPlayLoop(worker.model.engine, Game.DEVICE_ENV, cfg.max_moves,
                                       temperature_threshold=temperature_threshold,
                                       reward_scale=getattr(vec, "REWARD_SCALE", 1),
                                       first_game_id=worker.first_game_id, game_id_stride=worker.game_id_stride,
                                       td_steps=int(cfg.td_steps) if getattr(cfg, "PER", False) and getattr(cfg, "device_priorities", True) else 0,
                                       per_alpha=cfg.PER_alpha, discount=cfg.discount,
                                       staging_bytes=int(getattr(cfg, "selfplay_staging_bytes", 0) or 0))
        self.moves_per_call = int(getattr(cfg, "selfplay_moves_per_call", 64) or 64)   # upper bound of a chunk
        self.chunk = min(4, self.moves_per_call)                                      # adapted to the staging fill below
        self.device_ms = 0.0          # device time of all mz_selfplay_moves calls so far
        self.calls = 0
        self.parked_events = 0        # finished games that had to wait for a drain (staging area full), so far

    def moves(self, n_moves, temperature, **inject):
        """``n_moves`` lockstep moves -> ``PackedGames`` (a lazy sequence of the games that finished).  The moves run
        in chunks of ``moves_per_call`` per ``mz_selfplay_moves`` (one host synchronisation and one drain per chunk);
        if a chunk ever produces more finished games than the staging area holds, the surplus waits on the device
        (parked slots) and arrives with the next drain - nothing is lost."""
        out = PackedGames(self.obs_shape, self.obs_dtype, self.reward_type, self.loop.with_priorities)
        left = int(n_moves)
        if inject:                                   # parity / debug: one synchronous move with injected draws
            while left > 0:
                st = self.loop.moves(1, temperature, **inject)
                self._account(st, 1)
                out.add(*self.loop.drain())
                left -= 1
            return out
        # pipelined: while the host copies the games of chunk i out of one staging area, the device plays chunk i+1
        # into the other one (mz_selfplay_enqueue / wait; the library swaps the areas at every drain)
        k = min(left, self.chunk)
        self.loop.enqueue(k, temperature)
        left -= k
        while True:
            st = self.loop.wait()
            self._account(st, k)
            pointers = self.loop.drain_pointers()
            if left > 0:
                k = min(left, self.chunk)
                self.loop.enqueue(k, temperature)
                left -= k
                out.add(*self.loop.copy_staged(pointers))
            else:
                out.add(*self.loop.copy_staged(pointers))
                break
        return out

    def _account(self, st, k):
        self.device_ms += st.device_ms
        self.calls += 1
        self.parked_events += int(st.parked_slots)
        # next chunk: as many moves as fill about half of a staging area at the rate just seen, growing at most 2x per
        # call (the first finishes of a fresh batch arrive in a burst after a quiet start: one sample says little)
        if st.parked_slots:
            self.chunk = max(1, self.chunk // 2)
        else:
            grow = min(self.moves_per_call, 2 * max(k, 1))
            if st.staged_bytes > 0:
                grow = min(grow, int(0.5 * st.staging_capacity * k / st.staged_bytes))
            self.chunk = max(1, grow)


class PackedGames:
    """Finished games of one or more drains, still in their packed device format.  ``len``, iteration and indexing
    work like a list of ``GameHistory``; a ``PackedGameHistory`` is only created when an element is asked for, so
    handing thousands of games per second to a consumer costs nothing per game until the consumer looks at them
    (SURVEY.md 8f-2: bulk ingest with lazily materialised histories)."""

    def __init__(self, obs_shape, obs_dtype, reward_type, with_priorities=False):
        self._args = (obs_shape, obs_dtype, reward_type, with_priorities)
        self._chunks = []            # (bytes, index[n, 2])
        self._n = 0
        self.total_moves = 0

    def add(self, buf, index):
        if len(index):
            self._chunks.append((buf, index))
            self._n += len(index)
            self.total_moves += int((index[:, 1] & numpy.uint64(0xFFFFFFFF)).sum())

    def __len__(self):
        return self._n

    def __bool__(self):
        return self._n > 0

    def lengths(self):
        """Moves per game, without touching the blocks."""
        return numpy.concatenate([(ix[:, 1] & numpy.uint64(0xFFFFFFFF)).astype(numpy.int64) for _, ix in self._chunks]) \
            if self._chunks else numpy.zeros(0, numpy.int64)

    def _make(self, buf, off):
        return PackedGameHistory(parse_staged_game(buf, int(off)), *self._args)

    def blocks(self):
        """The games as ``parse_staged_game`` dicts (numpy views of the packed arrays), no history objects."""
        for buf, index in self._chunks:
            for off in index[:, 0]:
                yield parse_staged_game(buf, int(off))

    def __iter__(self):
        for buf, index in self._chunks:
            for off in index[:, 0]:
                yield self._make(buf, off)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        for buf, index in self._chunks:
            if i < len(index):
                return self._make(buf, index[i, 0])
            i -= len(index)
        raise IndexError("game index out of range")


class BatchedSelfPlay:
    """Lockstep self-play of B games: one ``mz_search`` call per move for the whole batch.

    Per move the host only (1) gathers observations / legal masks from the environments,
    (2) draws the root noise, (3) samples actions from the returned visit counts and
    (4) appends one struct-of-arrays record; ``GameHistory`` objects are materialised only when
    a game ends.  Game slot g has the global id ``first_game_id + g`` and draws from
    ``RandomState(seed + global id)``, so a game's history does not depend on how many games share the
    batch or on how many ranks the batch is split over (world-size invariance, SURVEY.md 8e).
    """

    def __init__(self, worker: SelfPlay, temperature, temperature_threshold, first_game_id=0):
        self.w = worker
        self.cfg = worker.config
        self.B = worker.num_parallel_games
        self.A = len(self.cfg.action_space)
        self.temperature = temperature
        self.temperature_threshold = temperature_threshold
        self.first_game_id = first_game_id
        Game = worker.Game
        if hasattr(Game, "vector"):
            self.env = Game.vector(self.B, worker.seed)
        else:
            self.env = _ObjectVector(Game, self.B, worker.seed, self.A)
        self.env_steps = 0                         # moves stepped by the batch so far (finished or not)
        self.numpy_mode = worker.rng_mode == "numpy"
        if self.numpy_mode:
            self.streams = [numpy.random.RandomState(worker.seed + first_game_id + g) for g in range(self.B)]
        else:
            self.fast = numpy.random.RandomState(worker.seed + first_game_id)

    def _noise_and_first(self, legal):
        cfg, B, A = self.cfg, self.B, self.A
        noise = numpy.zeros((B, A))
        if self.numpy_mode:
            first = numpy.zeros(B, numpy.int32)
            for g in range(B):
                idx = numpy.nonzero(legal[g])[0]
                noise[g, idx] = self.streams[g].dirichlet([cfg.root_dirichlet_alpha] * len(idx))
                first[g] = self.streams[g].choice(len(idx))
            return noise, first
        gam = self.fast.standard_gamma(cfg.root_dirichlet_alpha, size=(B, A)) * (legal > 0)
        noise = gam / gam.sum(1, keepdims=True)
        return noise, None

    def _actions(self, visit_counts, legal, moves_played):
        B = self.B
        actions = numpy.zeros(B, numpy.int64)
        thr = self.temperature_threshold
        if self.numpy_mode:
            for g in range(B):
                idx = numpy.nonzero(legal[g])[0]
                t = self.temperature if not thr or moves_played[g] + 1 < thr else 0
                actions[g] = _sample_action([int(a) for a in idx], visit_counts[g, idx].astype("int32"), t,
                                            self.streams[g])
            return actions
        t = numpy.full(B, float(self.temperature))
        if thr:
            t[moves_played + 1 >= thr] = 0
        greedy = t == 0
        with numpy.errstate(divide="ignore"):
            p = visit_counts.astype(numpy.float64) ** (1.0 / numpy.where(greedy, 1.0, t))[:, None]
        p = numpy.where(legal > 0, p, 0.0)           # 0 ** 0 = 1 at T = inf must not give illegal actions any mass
        cdf = numpy.cumsum(p / p.sum(1, keepdims=True), axis=1)
        u = self.fast.random_sample(B)
        last_legal = self.A - 1 - numpy.argmax(legal[:, ::-1] > 0, axis=1)
        sampled = numpy.minimum((u[:, None] >= cdf).sum(1), last_legal)    # cdf rounding can leave u >= cdf[-1]
        return numpy.where(greedy, numpy.where(legal > 0, visit_counts, -1).argmax(1), sampled).astype(numpy.int64)

    def _begin(self):
        B = self.B
        env = self.env
        self.obs = env.reset()
        # per-slot bookkeeping
        self.start = numpy.zeros(B, numpy.int64)        # index into `records` of the slot's first move
        self.moves = numpy.zeros(B, numpy.int64)        # moves played in the current game
        self.first_obs = [numpy.asarray(self.obs[g]).copy() for g in range(B)]
        self.first_to_play = numpy.asarray(env.to_play()).copy()
        self.game_ids = (self.first_game_id + numpy.arange(B)).astype(numpy.int64)
        self.records = deque()                          # one dict of [B,...] arrays per move
        self.base = 0                                   # absolute index of records[0]
        self.t_abs = 0
        self._begun = True

    def move(self):
        """One lockstep move of the whole batch; returns the GameHistory objects of the games it finished."""
        if not getattr(self, "_begun", False):
            self._begin()
        cfg, B, A, w = self.cfg, self.B, self.A, self.w
        env, records, start, moves, first_obs = self.env, self.records, self.start, self.moves, self.first_obs
        engine = w.model.engine
        obs = self.obs
        legal = numpy.asarray(env.legal_mask(), dtype=numpy.uint8)
        to_play = numpy.asarray(env.to_play(), dtype=numpy.int32)
        if cfg.stacked_observations:
            batch = numpy.stack([self._stacked(g, obs, records, self.base, start, first_obs) for g in range(B)])
        else:
            batch = numpy.stack([numpy.asarray(o, dtype=numpy.float32) for o in obs]) \
                if not isinstance(obs, numpy.ndarray) else obs
        noise, first = self._noise_and_first(legal)
        out = engine.search(obs=numpy.asarray(batch, dtype=numpy.float32).reshape(B, -1), legal_mask=legal,
                            to_play=to_play, add_exploration_noise=True, noise=noise, first_index=first,
                            game_id=self.game_ids, move_index=moves.astype(numpy.int32))
        actions = self._actions(out.visit_counts, legal, moves)
        obs, reward, done = env.step(actions)
        records.append(dict(visits=out.visit_counts, legal=legal, root_value=out.root_value, action=actions,
                            obs=[numpy.asarray(o).copy() for o in obs] if not isinstance(obs, numpy.ndarray) else obs.copy(),
                            reward=numpy.asarray(reward).copy() if isinstance(reward, numpy.ndarray) else list(reward),
                            to_play=numpy.asarray(env.to_play()).copy()))
        self.t_abs += 1
        moves += 1
        self.env_steps += B
        out_games = []
        finished = numpy.asarray(done, dtype=bool) | (moves >= cfg.max_moves)
        if finished.any():
            for g in numpy.nonzero(finished)[0]:
                gh = self._materialise(g, records, self.base, int(start[g]), self.t_abs, first_obs[g], self.first_to_play[g])
                w.played_games += 1                  # counted when the game is handed over, like self_play.py:52
                w.played_steps += len(gh.action_history) - 1
                out_games.append(gh)
            obs = env.reset(finished)
            tp = numpy.asarray(env.to_play())
            for g in numpy.nonzero(finished)[0]:
                first_obs[g] = numpy.asarray(obs[g]).copy()
                self.first_to_play[g] = tp[g]
                start[g] = self.t_abs
                moves[g] = 0
                self.game_ids[g] += w.game_id_stride       # a fresh global game id for the slot's next game
                if self.numpy_mode:
                    self.streams[g] = numpy.random.RandomState(self.w.seed + int(self.game_ids[g]))
        self.obs = obs
        drop = int(start.min()) - self.base
        for _ in range(drop):
            records.popleft()
        self.base += drop
        return out_games

    def run(self):
        """Generator over finished games, one lockstep move at a time."""
        while True:
            for gh in self.move():
                yield gh

    def _stacked(self, g, obs, records, base, start, first_obs):
        gh = GameHistory()
        gh.observation_history.append(first_obs[g])
        gh.action_history.append(0)
        for r in list(records)[int(start[g]) - base:]:
            gh.observation_history.append(numpy.asarray(r["obs"][g]))
            gh.action_history.append(r["action"][g])
        return gh.get_stacked_observations(-1, self.cfg.stacked_observations, self.A)

    def _materialise(self, g, records, base, first, last, obs0, to_play0):
        """Column g of the per-move records [first, last) -> one reference-format GameHistory."""
        cfg = self.cfg
        gh = GameHistory()
        gh.action_history.append(0)
        gh.observation_history.append(obs0)
        gh.reward_history.append(0)
        gh.to_play_history.append(int(to_play0))
        for i in range(first - base, last - base):
            r = records[i]
            gh.store_visit_counts(r["visits"][g], r["legal"][g], r["root_value"][g], cfg.action_space)
            gh.action_history.append(r["action"][g])
            gh.observation_history.append(numpy.asarray(r["obs"][g]))
            rew = r["reward"][g]
            gh.reward_history.append(rew.item() if hasattr(rew, "item") else rew)
            gh.to_play_history.append(int(r["to_play"][g]))
        return gh
