"""Evaluation games on the CPU (search supplied by the oracle-backed test double): histories with opponent moves,
the summary statistics of the reference's test worker and MuZero.test, the host path of SelfPlay.play_test_games,
the test-mode report and the opponent / muzero_player arguments."""
import warnings

import numpy
import pytest
import torch

from conftest import weights_for
from eval_helpers import pack_block
from fake_engine import FakeSearchEngine
from muzero_general_b200 import self_play as sp
from muzero_general_b200.games import load_game_module
from muzero_general_b200.netspec import netspec_from_config

torch.set_num_threads(1)


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(sp, "SearchEngine", FakeSearchEngine)


def _worker(name, seed=0, **over):
    mod = load_game_module(name)
    cfg = mod.MuZeroConfig()
    for k, v in over.items():
        setattr(cfg, k, v)
    return sp.SelfPlay({"weights": weights_for(name, netspec_from_config(cfg))}, mod.Game, cfg, seed), cfg


def _reference_report(h, muzero_player, players):
    """self_play.py:67-90 and muzero.py:411-424 for one GameHistory, as the reference writes them."""
    with warnings.catch_warnings():                 # numpy.mean([]) warns and gives NaN
        warnings.simplefilter("ignore")
        mean_value = numpy.mean([value for value in h.root_values if value])
    out = {"episode_length": len(h.action_history) - 1, "total_reward": sum(h.reward_history), "mean_value": mean_value}
    if players > 1:
        out["muzero_reward"] = sum(reward for i, reward in enumerate(h.reward_history)
                                   if h.to_play_history[i - 1] == muzero_player)
        out["opponent_reward"] = sum(reward for i, reward in enumerate(h.reward_history)
                                     if h.to_play_history[i - 1] != muzero_player)
        out["result"] = out["muzero_reward"]
    else:
        out["result"] = sum(h.reward_history)
    return out


def _history(actions, rewards, to_play, root_values, visits, first_to_play=0):
    h = sp.GameHistory()
    h.action_history = [0] + list(actions)
    h.reward_history = [0] + list(rewards)
    h.to_play_history = [first_to_play] + list(to_play)
    h.root_values = list(root_values)
    h.child_visits = [list(v) for v in visits]
    h.observation_history = [numpy.zeros((3, 3, 3))] * (len(actions) + 1)
    return h


def _same(a, b):
    return (numpy.isnan(a) and numpy.isnan(b)) if isinstance(a, float) and numpy.isnan(a) else a == b


def test_packed_block_with_opponent_rows_materialises_like_the_reference():
    """Opponent rows (root value NaN, zero visits) become what store_search_statistics(None, ...) leaves: None in
    root_values and no child_visits row; searched rows are normalised visit counts; the summary read from the packed
    arrays equals the one computed from the materialised histories."""
    rs = numpy.random.RandomState(0)
    A, O, T = 9, 27, 7
    blocks, refs = [], []
    for gid, first_player_is_muzero in ((3, True), (4, False)):
        searched = numpy.array([(t % 2 == 0) == first_player_is_muzero for t in range(T)])
        visits = numpy.where(searched[:, None], rs.randint(0, 5, (T, A)), 0).astype(numpy.int32)
        visits[searched, 0] += 1
        root = numpy.where(searched, rs.standard_normal(T), numpy.nan)
        action = rs.randint(0, A, T)
        reward = numpy.zeros(T, numpy.float32)
        reward[-1] = 20.0
        to_play = numpy.array([(t + 1) % 2 for t in range(T)], numpy.int32)
        obs = rs.randint(0, 2, (T + 1, O)).astype(numpy.float32)
        blocks.append(pack_block(gid, gid % 2, 0, root, visits, action, reward, to_play, obs))
        ref = sp.GameHistory()
        ref.action_history, ref.reward_history, ref.to_play_history = [0], [0], [0]
        ref.observation_history = [obs[0].reshape(3, 3, 3).astype(numpy.int32)]
        for t in range(T):
            if searched[t]:
                total = visits[t].sum()
                ref.child_visits.append([visits[t, a] / total for a in range(A)])
                ref.root_values.append(float(root[t]))
            else:
                ref.root_values.append(None)
            ref.action_history.append(int(action[t]))
            ref.observation_history.append(obs[t + 1].reshape(3, 3, 3).astype(numpy.int32))
            ref.reward_history.append(int(reward[t]))
            ref.to_play_history.append(int(to_play[t]))
        refs.append(ref)
    buf = b"".join(blocks)
    index = numpy.array([[0, (0 << 32) | T], [len(blocks[0]), (1 << 32) | T]], numpy.uint64)
    games = sp.PackedGames((3, 3, 3), numpy.int32, int)
    games.add(buf, index)
    hist = list(games)
    for gh, ref in zip(hist, refs):
        assert gh.root_values == ref.root_values
        assert gh.child_visits == ref.child_visits
        assert gh.action_history == ref.action_history and gh.reward_history == ref.reward_history
        assert gh.to_play_history == ref.to_play_history
        assert all(numpy.array_equal(a, b) for a, b in zip(gh.observation_history, ref.observation_history))
        assert len(gh.child_visits) == sum(v is not None for v in gh.root_values)
    for mp in (0, 1):
        packed, listed = sp.evaluation_summary(games, 2, mp), sp.evaluation_summary(hist, 2, mp)
        assert packed.keys() == listed.keys()
        assert all(_same(packed[k], listed[k]) for k in packed), (packed, listed)


def test_summary_equals_the_reference_formulas():
    """Per game the reference's test-worker keys and MuZero.test's result; over games their average, with W/D/L from
    muzero vs opponent reward.  A game whose root values are all 0.0 or None has a NaN mean value (the reference's
    numpy.mean of an empty list) and stays out of that average."""
    games = [
        _history([4, 0, 1, 3, 2], [0, 0, 0, 0, 20], [1, 0, 1, 0, 1], [0.5, None, -0.25, None, 0.75], [[1] * 9] * 3),
        _history([0, 4, 1, 8], [0, 0, 0, 20], [1, 0, 1, 0], [None, 0.0, None, 0.0], [[1] * 9] * 2),        # all 0 / None
        _history([0, 1, 2], [0, 0, 0], [1, 0, 1], [0.125, None, 0.375], [[1] * 9] * 2),
    ]
    for mp in (0, 1):
        per_game = [_reference_report(h, mp, 2) for h in games]
        assert numpy.isnan(per_game[1]["mean_value"])
        s = sp.evaluation_summary(games, 2, mp)
        assert s["num_games"] == 3
        for k in ("episode_length", "total_reward", "muzero_reward", "opponent_reward", "result"):
            assert s[k] == numpy.mean([r[k] for r in per_game]), k
        assert s["mean_value"] == numpy.mean([r["mean_value"] for r in per_game if not numpy.isnan(r["mean_value"])])
        wins = sum(r["muzero_reward"] > r["opponent_reward"] for r in per_game)
        losses = sum(r["muzero_reward"] < r["opponent_reward"] for r in per_game)
        assert (s["wins"], s["draws"], s["losses"]) == (wins, 3 - wins - losses, losses)
        for h, r in zip(games, per_game):                    # one game: exactly the reference's numbers
            one = sp.evaluation_summary([h], 2, mp)
            assert all(_same(float(one[k]), float(r[k])) for k in r), (one, r)
    one_player = sp.evaluation_summary(games, 1, 0)
    assert one_player["result"] == numpy.mean([sum(h.reward_history) for h in games])
    assert "muzero_reward" not in one_player and "wins" not in one_player


@pytest.mark.parametrize("opponent,muzero_player", [("expert", 0), ("expert", 1), ("random", 1)])
def test_host_path_searches_exactly_muzero_moves(opponent, muzero_player, fake_engine):
    worker, cfg = _worker("tictactoe", num_simulations=4)
    assert worker.loop_path == "host"
    games, summary = worker.play_test_games(3, opponent, muzero_player)
    assert len(games) == 3 and summary["num_games"] == 3
    for h in games:
        T = len(h.action_history) - 1
        assert T <= cfg.max_moves and len(h.root_values) == T and h.to_play_history[0] == 0
        mine = [h.to_play_history[t] == muzero_player for t in range(T)]
        assert [v is not None for v in h.root_values] == mine
        assert len(h.child_visits) == sum(mine)
    assert summary["wins"] + summary["draws"] + summary["losses"] == 3


def test_test_mode_reports_averages_over_test_games_per_report(fake_engine):
    worker, cfg = _worker("tictactoe", num_simulations=3, training_steps=4)
    cfg.test_games_per_report = 2

    class Storage:
        def __init__(self):
            self.d = dict(weights=weights_for("tictactoe", netspec_from_config(cfg)), training_step=0, terminate=False)
            self.writes = []

        def get_info(self, k):
            if k == "training_step":
                self.d["training_step"] += 1
            return self.d[k]

        def set_info(self, k, v=None):
            self.writes.append(k)
            self.d.update(k)

    storage = Storage()
    worker.continuous_self_play(storage, None, test_mode=True)
    keys = set().union(*storage.writes)
    assert keys == {"episode_length", "total_reward", "mean_value", "muzero_reward", "opponent_reward"}
    reports = len(storage.writes) // 2
    assert reports >= 1 and worker.played_games == 2 * reports
    assert 5 <= storage.d["episode_length"] <= 9 and worker._next_test_game_id == worker.played_games


def test_opponent_arguments():
    ttt = load_game_module("tictactoe").MuZeroConfig()
    ttt.muzero_player = 1
    assert sp.resolve_opponent(ttt) == ("expert", 1)
    assert sp.resolve_opponent(ttt, "random", 0) == ("random", 0)           # an explicit 0 is not replaced
    assert sp.resolve_opponent(ttt, None, 0) == ("expert", 0)
    with pytest.raises(ValueError):
        sp.resolve_opponent(ttt, "human")
    with pytest.raises(ValueError):
        sp.resolve_opponent(ttt, "minimax")
    cartpole = load_game_module("cartpole").MuZeroConfig()
    assert sp.resolve_opponent(cartpole, "expert", 0) == ("self", 0)
    assert sp.resolve_opponent(cartpole) == ("self", 0)
