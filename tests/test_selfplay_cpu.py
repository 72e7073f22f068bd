"""Host-side self-play logic on the CPU (search supplied by the oracle-backed test double):
draw order, GameHistory format, batched lockstep play, the training batch the reference's own
ReplayBuffer builds from our histories (recorded golden data)."""
import pickle

import numpy
import pytest
import torch

from conftest import golden_json, weights_for
from fake_engine import FakeSearchEngine
from muzero_general_b200 import self_play as sp
from muzero_general_b200.games import load_game_module
from muzero_general_b200.netspec import netspec_from_config

torch.set_num_threads(1)


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(sp, "SearchEngine", FakeSearchEngine)


def _worker(name, seed, **over):
    mod = load_game_module(name)
    cfg = mod.MuZeroConfig()
    for k, v in over.items():
        setattr(cfg, k, v)
    spec = netspec_from_config(cfg)
    return sp.SelfPlay({"weights": weights_for(name, spec)}, mod.Game, cfg, seed), cfg


def _assert_history_equals(gh, ref):
    assert [int(a) for a in gh.action_history] == ref["action_history"]
    assert [float(r) for r in gh.reward_history] == ref["reward_history"]
    assert [int(t) for t in gh.to_play_history] == ref["to_play_history"]
    assert [[float(x) for x in c] for c in gh.child_visits] == ref["child_visits"]
    assert [float(v) for v in gh.root_values] == ref["root_values"]           # fp64 equality
    assert [numpy.asarray(o).astype(float).ravel().tolist() for o in gh.observation_history] == ref["observation_history"]


def test_env_fixtures():
    """Our board environments replay the reference's recorded trajectories."""
    for name in ("tictactoe", "connect4", "gomoku"):
        fx = golden_json(f"env_{name}.json")
        mod = load_game_module(name)
        for steps in fx["games"]:
            g = mod.Game(0)
            g.reset()
            for s in steps:
                obs, reward, done = g.step(s["action"])
                assert str(obs.dtype) == fx["obs_dtype"]
                assert obs.astype(numpy.int8).ravel().tolist() == s["obs"]
                assert (reward, done, g.to_play(), g.legal_actions()) == (s["reward"], s["done"], s["to_play"], s["legal"])


@pytest.mark.parametrize("name", ["tictactoe", "connect4"])
def test_play_game_reproduces_reference_games(name, fake_engine):
    """Same weights, same legacy numpy seed -> the reference's GameHistory, value for value."""
    for ref in golden_json("play.json")[name]:
        worker, cfg = _worker(name, ref["seed"], num_simulations=ref["num_simulations"])
        gh = worker.play_game(ref["temperature"], cfg.temperature_threshold, False, "self", 0)
        _assert_history_equals(gh, ref)
        assert gh.action_history[0] == 0 and isinstance(gh.root_values[0], float)
        assert all(isinstance(x, (float, int)) for x in gh.child_visits[0])


def test_mcts_run_returns_reference_shaped_tree(fake_engine):
    worker, cfg = _worker("tictactoe", 0)
    c = golden_json("mcts_tictactoe.json")[0]
    numpy.random.seed(c["seed"])
    obs = numpy.array(c["obs"]).reshape(c["obs_shape"])
    root, info = sp.MCTS(cfg).run(worker.model, obs, c["legal"], c["to_play"], True)
    assert list(root.children.keys()) == c["root_actions"]
    assert [root.children[a].visit_count for a in c["root_actions"]] == c["root_visits"]
    assert [root.children[a].prior for a in c["root_actions"]] == c["root_priors"]
    assert [root.children[a].value_sum for a in c["root_actions"]] == c["root_child_value_sums"]
    assert root.value() == c["root_value"] and root.visit_count == c["num_simulations"]
    assert info == {"max_tree_depth": c["max_tree_depth"], "root_predicted_value": c["root_predicted_value"]}
    # walk the first recorded path: every node on it is expanded, with hidden state and reward
    node = root
    for a in c["sims"][-1]["actions"][:-1]:
        node = node.children[a]
        assert node.expanded() and node.hidden_state is not None and node.to_play in (0, 1)
    assert sp.SelfPlay.select_action(root, 0) == c["root_actions"][int(numpy.argmax(c["root_visits"]))]


def test_batched_play_is_batch_size_invariant(fake_engine):
    """Game slot g draws from RandomState(seed+g): its history does not depend on the batch."""
    worker4, _ = _worker("tictactoe", 3, num_parallel_games=4, num_simulations=10)
    games4 = worker4.play_games(4, 1.0)
    assert len(games4) >= 4
    worker1, _ = _worker("tictactoe", 3, num_parallel_games=1, num_simulations=10)
    solo = worker1.play_games(1, 1.0)[0]
    # slot 0 of the batch of four is the same game as the batch of one
    first = [g for g in games4 if len(g.action_history) == len(solo.action_history)
             and [int(a) for a in g.action_history] == [int(a) for a in solo.action_history]]
    assert first, "slot 0's game not found in the larger batch"
    assert first[0].root_values == solo.root_values and first[0].child_visits == solo.child_visits
    for g in games4:
        T = len(g.action_history) - 1
        assert len(g.child_visits) == T == len(g.root_values) and len(g.observation_history) == T + 1
        assert all(abs(sum(c) - 1) < 1e-12 for c in g.child_visits)


def test_fast_rng_mode_and_max_moves(fake_engine):
    worker, cfg = _worker("cartpole", 0, num_parallel_games=3, num_simulations=4, rng_mode="philox", max_moves=5)
    games = worker.play_games(3, 1.0)
    for g in games:
        assert 1 <= len(g.action_history) - 1 <= 5
        assert g.observation_history[0].shape == (1, 1, 4) and g.reward_history[1] == 1.0


def test_our_histories_give_the_reference_replay_buffer_batch(fake_engine):
    """GameHistory objects produced by this package, passed through pickle (the Ray boundary), yield the training
    batch the unmodified reference ReplayBuffer.save_game / get_batch built from the same games (SURVEY.md 8c
    'consumer acceptance'; recorded in tests/golden/replay_buffer.json by oracle/gen_golden.py --replay): the
    priorities it attached, and at every sampled position the stacked observation and, for each unroll step inside
    the game, the target value, reward, policy and action."""
    from muzero_general_b200 import reanalyse as ra
    want = golden_json("replay_buffer.json")["batch"]
    worker, cfg = _worker("tictactoe", 1, num_parallel_games=4, num_simulations=8)
    games = [pickle.loads(pickle.dumps(gh)) for gh in worker.play_games(6, 1.0)]
    assert len(games) == want["num_games"]
    for gh, pri, top in zip(games, want["priorities"], want["game_priority"]):
        mine, mine_top = ra.initial_priorities(gh, cfg)
        assert numpy.array_equal(mine, numpy.array(pri, numpy.float32)) and mine_top == top
    assert len(want["index"]) == 8
    for row, (g, pos) in enumerate(want["index"]):
        gh = games[g]
        obs = gh.get_stacked_observations(pos, cfg.stacked_observations, len(cfg.action_space))
        assert numpy.asarray(obs, dtype=numpy.float64).ravel().tolist() == want["observation"][row]
        values = ra.target_values(gh, cfg)
        for k in range(cfg.num_unroll_steps + 1):
            i = pos + k
            if i >= len(gh.root_values):
                break
            assert float(values[i]) == want["value"][row][k], (row, k)
            assert float(gh.reward_history[i]) == want["reward"][row][k]
            assert [float(p) for p in gh.child_visits[i]] == want["policy"][row][k]
            assert int(gh.action_history[i]) == want["action"][row][k]


class _Storage:
    """Plain-object stand-in for shared_storage.SharedStorage (get_info / set_info, shared_storage.py:23-40)."""

    def __init__(self, weights, training_steps_per_poll=1):
        self.d = dict(weights=weights, training_step=0, terminate=False, num_played_steps=0, num_played_games=0)
        self.polls = 0
        self.rate = training_steps_per_poll

    def get_info(self, keys):
        if keys == "training_step":          # pretend a trainer is making progress while we play
            self.polls += 1
            self.d["training_step"] += self.rate
        return self.d[keys] if isinstance(keys, str) else {k: self.d[k] for k in keys}

    def set_info(self, keys, values=None):
        if isinstance(keys, dict):
            self.d.update(keys)
        else:
            self.d[keys] = values


class _Buffer:
    def __init__(self):
        self.games = []

    def save_game(self, game_history, shared_storage=None):
        self.games.append(game_history)
        if shared_storage is not None:
            shared_storage.set_info("num_played_games", len(self.games))
            shared_storage.set_info("num_played_steps", sum(len(g.root_values) for g in self.games))


@pytest.mark.parametrize("parallel", [1, 3])
def test_continuous_self_play_loop(parallel, fake_engine):
    """The actor loop of self_play.py:31-108 with plain objects in place of the Ray handles: refreshes the
    weights, plays until training_steps is reached, pushes every finished game to the buffer."""
    worker, cfg = _worker("tictactoe", 0, num_parallel_games=parallel, num_simulations=5, training_steps=12, ratio=None)
    storage = _Storage(weights_for("tictactoe", netspec_from_config(cfg)), training_steps_per_poll=2)
    buf = _Buffer()
    worker.continuous_self_play(storage, buf)
    assert buf.games and all(len(g.child_visits) == len(g.action_history) - 1 for g in buf.games)
    assert storage.d["num_played_games"] == len(buf.games)
    assert storage.d["training_step"] >= cfg.training_steps


def test_continuous_self_play_test_mode_reports_metrics(fake_engine):
    """test_mode: greedy play, metrics written to the shared storage (self_play.py:54-90)."""
    worker, cfg = _worker("tictactoe", 0, num_simulations=5, training_steps=6, opponent="random", muzero_player=0)
    storage = _Storage(weights_for("tictactoe", netspec_from_config(cfg)), training_steps_per_poll=3)
    worker.continuous_self_play(storage, _Buffer(), test_mode=True)
    for key in ("episode_length", "total_reward", "mean_value", "muzero_reward", "opponent_reward"):
        assert key in storage.d
    assert 5 <= storage.d["episode_length"] <= 9


@pytest.mark.parametrize("name", ["tictactoe", "connect4"])
def test_expert_agent_matches_reference(name):
    """The hard-coded evaluation opponent (games/*.py expert_action) picks the reference's move at every position
    of the recorded playouts, consuming the global numpy stream the same way."""
    mod = load_game_module(name)
    cases = golden_json("expert.json")[name]
    assert len(cases) > 100
    for c in cases:
        g = mod.Game(0)
        g.reset()
        for a in c["moves"]:
            g.step(a)
        numpy.random.seed(c["seed"])
        assert int(g.expert_agent()) == c["action"], c


def test_test_mode_with_the_shipped_default_opponent(fake_engine):
    """The shipped board-game configs keep opponent="expert" (games/tictactoe.py, games/connect4.py): the evaluation
    worker must run with them as they are."""
    for name in ("tictactoe", "connect4"):
        worker, cfg = _worker(name, 0, num_simulations=4, training_steps=6)
        assert cfg.opponent == "expert"
        storage = _Storage(weights_for(name, netspec_from_config(cfg)), training_steps_per_poll=3)
        worker.continuous_self_play(storage, _Buffer(), test_mode=True)
        assert storage.d["episode_length"] >= 5 and "opponent_reward" in storage.d


@pytest.mark.parametrize("name,mode", [("tictactoe", "numpy"), ("cartpole", "numpy"), ("cartpole", "philox")])
def test_consecutive_batches_are_new_games(name, mode, fake_engine):
    """play_games keeps ONE lockstep batch alive across calls: new start states / RNG streams / game ids every game,
    games in flight at the end of a call are finished by the next one, counters count handed-over games."""
    worker, cfg = _worker(name, 0, num_parallel_games=3, num_simulations=4, rng_mode=mode, max_moves=12)
    first = worker.play_games(3, 1.0)
    ids_after_first = worker._batched.game_ids.copy()
    steps_first = worker._batched.env_steps
    second = worker.play_games(3, 1.0)
    assert len(first) == 3 and len(second) == 3
    key = lambda g: ([int(a) for a in g.action_history], [numpy.asarray(o).tobytes() for o in g.observation_history],
                     g.child_visits)
    assert all(key(a) != key(b) for a in first for b in second)
    assert len({tuple(key(g)[0]) + (key(g)[1][0],) for g in first + second}) >= 4
    assert (worker._batched.game_ids >= ids_after_first).all() and worker._batched.game_ids.max() >= 3
    assert worker._batched.env_steps > steps_first
    assert worker.played_games == 6
    assert worker.played_steps == sum(len(g.action_history) - 1 for g in first + second)
    # a different temperature applies from the next move on, without restarting the batch
    batch = worker._batched
    worker.play_games(1, 0.0)
    assert worker._batched is batch and batch.temperature == 0.0


def test_long_games_survive_the_quota(fake_engine):
    """Short games recycle their slots while a long game is in flight; the long one is still delivered later."""
    worker, cfg = _worker("cartpole", 0, num_parallel_games=4, num_simulations=3, rng_mode="philox", max_moves=40)
    lengths = []
    for _ in range(6):
        lengths += [len(g.action_history) - 1 for g in worker.play_games(2, 1.0)]
    assert worker.played_games == 12 and len(lengths) == 12
    assert sum(lengths) == worker.played_steps <= worker._batched.env_steps


def test_search_rejects_a_row_without_legal_actions():
    from muzero_general_b200.engine import SearchEngine
    eng = SearchEngine.__new__(SearchEngine)          # marshalling only: no library / GPU needed for the check
    eng.A, eng.N, eng.obs_elems = 3, 2, 4
    with pytest.raises(AssertionError, match="Legal actions should not be an empty array"):
        eng.search(obs=numpy.zeros((2, 4), numpy.float32), legal_mask=numpy.array([[1, 0, 0], [0, 0, 0]], numpy.uint8))
